"""TEST INFRASTRUCTURE ONLY -- the oracle of tests/test_resume_oracle.py and tests/test_gpu_resume.py.

`ResumeOracle(flat)` is the restart-set oracle (tests/restart_oracle.py: the CPU oracle's graph, rankings and restart sets)
plus a stateful Model: `rank` starts from any vector and a sequence of run(int) / run(double) / run() calls follows, each
from the rank the previous one left (tests/resume_oracle.cpp, compiled on first use into a temporary directory)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from restart_oracle import RestartOracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        d = tempfile.mkdtemp(prefix="resume_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libresume_oracle.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                               "-o", so, os.path.join(_HERE, "resume_oracle.cpp")])
        L = C.CDLL(so)
        vp, i32, f64 = C.c_void_p, C.c_int32, C.c_double
        L.rs_run.argtypes = [i32, vp, vp, vp, f64, vp, vp, vp, i32, i32, vp, vp, vp, i32, vp, vp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def fixed(n: int):
    """run(int n)"""
    return (0, int(n), 0.0)


def threshold(thr: float, max_iter: int = 0):
    """run(double thr); max_iter > 0 bounds it"""
    return (1, int(max_iter), float(thr))


def default_threshold(max_iter: int = 0):
    """run()"""
    return (2, int(max_iter), 0.0)


class ResumeOracle(RestartOracle):
    def constructor_rank(self, seed: int) -> np.ndarray:
        """Model.cs:24 (seed -1) / :44"""
        if seed < 0:
            return np.ones(self.n)
        r = np.zeros(self.n)
        r[seed] = float(self.n)
        return r

    def run_ops(self, rank0, ops, damping: float, seed: int | None = None, nodes=None, weights=None, literal: bool = False):
        """A Model with `rank` = rank0 and the restart vector of `seed` (one-hot; -1: uniform) or of `weights` at `nodes`,
        then `ops` (fixed / threshold / default_threshold) -> (rank[N], deliverRanks() calls per op)."""
        if nodes is None:
            if seed is None or seed < 0:
                nodes, weights = np.zeros(0, np.int32), np.zeros(0)
            else:
                nodes, weights = [seed], [1.0]
        nodes = np.ascontiguousarray(nodes, np.int32)
        weights = np.ascontiguousarray(weights, np.float64)
        rank0 = np.ascontiguousarray(rank0, np.float64)
        assert rank0.shape == (self.n,)
        kind = np.ascontiguousarray([o[0] for o in ops], np.int32)
        count = np.ascontiguousarray([o[1] for o in ops], np.int64)
        thr = np.ascontiguousarray([o[2] for o in ops], np.float64)
        rank = np.empty(max(self.n, 1), np.float64)
        iters = np.zeros(max(len(ops), 1), np.int64)
        rc = lib().rs_run(self.n, _p(self.rp), _p(self.col), _p(self.val), float(damping), _p(rank0), _p(nodes), _p(weights),
                          len(nodes), len(ops), _p(kind), _p(count), _p(thr), int(literal), _p(rank), _p(iters))
        if rc < 0:
            raise ValueError("rs_run: bad argument")
        return rank[:self.n], iters[:len(ops)].tolist()
