"""CPU tests of the resume oracle (tests/resume_oracle.cpp): a Model started from any rank -- the constructor's or one the
caller wrote -- then a sequence of run(int) / run(double) / run() calls, each from the rank the previous one left.  Its
collapsed and literal forms against the pure-Python restatement (oracle/rwr_literal.py) with `model.rank` assigned, and,
from the constructor state, against the seeded oracle (liboracle) and the restart-set oracle."""
import random

import numpy as np
import pytest

from conftest import bits, load_golden
from random_graphs import random_flat
import oracle as O
import rwr_literal as R
from resume_oracle import ResumeOracle, fixed, threshold

C015 = O.widen_float(0.15)


def same(a, b):
    """bit for bit, except that any NaN equals any NaN (the payload of a NaN differs between C++ and Python arithmetic)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(a[~na]), bits(b[~nb]))


def literal_of(flat):
    pg = R.graph_from_flat(flat["node_id"], flat["node_type"], flat["src"], flat["dst"], flat["etype"], flat["w"])
    pg.buildGraph()
    return pg


def python_run(pg, n, rank0, ops, seed=None, nodes=None, weights=None):
    """rwr_literal's Model with `rank` (and, for a node set, `restart`) assigned, then the same calls"""
    m = R.Model(pg, C015, seed) if seed is not None and seed >= 0 else R.Model(pg, C015)
    if nodes is not None:
        q = [0.0] * n
        for v, w in zip(nodes, weights):
            q[v] = float(w)
        m.restart = q
    m.rank = [float(x) for x in rank0]
    iters = []
    for kind, count, thr in ops:
        d0 = m.nDeliver
        if kind == 0:
            m.run(count)
        elif kind == 1:
            m.run(thr)
        else:
            m.run()
        iters.append(m.nDeliver - d0)
    return np.array(m.rank), iters


def starts(rng, og, seed):
    """the constructor's rank, a random positive vector, one with exact zeros"""
    n = og.n
    pos = np.array([rng.random() * 2 + 1e-3 for _ in range(n)])
    zeros = pos.copy()
    zeros[rng.sample(range(n), n // 2)] = 0.0
    return [og.constructor_rank(seed), pos, zeros]


def check(og, pg, rank0, ops, **restart):
    a, ia = og.run_ops(rank0, ops, C015, literal=True, **restart)
    b, ib = og.run_ops(rank0, ops, C015, literal=False, **restart)
    assert ia == ib and np.array_equal(bits(a), bits(b)), ("collapsed", ops, restart)
    p, ip = python_run(pg, og.n, rank0, ops, **restart)
    assert ia == ip and same(a, p), ("python", ops, restart)
    return a, ia


FIXED_SEQS = [[fixed(3), fixed(4)], [fixed(1), fixed(1), fixed(5)], [fixed(0), fixed(2)]]
THR_SEQS = [[fixed(2), threshold(1e-6)], [threshold(1e-3), fixed(3), threshold(1e-9)], [fixed(5), threshold(1e-12)]]


def cases(rng, flat, poison):
    og, pg = ResumeOracle(flat), literal_of(flat)
    n = og.n
    seed = rng.randrange(n)
    nodes = rng.sample(range(n), min(3, n))
    weights = [0.5, 0.25, 0.25][:len(nodes)]
    for restart in (dict(seed=seed), dict(seed=-1), dict(nodes=nodes, weights=weights)):
        s = restart.get("seed", -1)
        for rank0 in starts(rng, og, s):
            for ops in FIXED_SEQS + ([] if poison else THR_SEQS):
                check(og, pg, rank0, ops, **restart)


@pytest.mark.parametrize("gseed", [11, 12, 13, 14])
def test_resumed_runs_equal_the_literal_model_on_random_graphs(gseed):
    """dangling rows, multi-edges and (odd seeds) NaN / Inf rows; one-hot, uniform and node-set restart vectors"""
    rng = random.Random(gseed)
    poison = gseed % 2 == 1
    flat = random_flat(rng, 8, 20, 3, 90, zero_rows=1 if poison else 0, nan_rows=1 if poison else 0)
    cases(rng, flat, poison)


@pytest.mark.parametrize("name", ["kat_8c", "small_a", "small_b"])
def test_resumed_runs_equal_the_literal_model_on_the_golden_graphs(name):
    cases(random.Random(name), load_golden(name)["input"], False)


def test_written_nan_and_inf_ranks_poison_like_the_literal_model():
    rng = random.Random(7)
    flat = random_flat(rng, 8, 20, 3, 90)
    og, pg = ResumeOracle(flat), literal_of(flat)
    for bad in (np.nan, np.inf, -np.inf):
        rank0 = np.ones(og.n)
        rank0[rng.randrange(og.n)] = bad
        for restart in (dict(seed=0), dict(seed=-1), dict(nodes=[1, 2], weights=[0.5, 0.5])):
            a, _ = check(og, pg, rank0, [fixed(1), fixed(2)], **restart)
            assert np.isnan(a).all(), (bad, restart)


@pytest.mark.parametrize("gseed", [21, 22])
def test_constructor_starts_equal_the_seeded_and_the_restart_set_oracles(gseed):
    """run(a) then run(b) from the constructor state is run(a + b) of liboracle (seeded) and of the restart-set oracle;
    run(a) then run(thr) matches the restart-set oracle's iteration when the initial rank is the one run(a) left"""
    rng = random.Random(gseed)
    flat = random_flat(rng, 8, 20, 3, 90, zero_rows=1, nan_rows=0)
    og = ResumeOracle(flat)
    for s in rng.sample(range(og.n), 4):
        for a, b in ((0, 1), (1, 1), (2, 3), (5, 15)):
            got, it = og.run_ops(og.constructor_rank(s), [fixed(a), fixed(b)], C015, seed=s)
            want, _ = og.run(s, C015, n_iter=a + b)
            assert it == [a, b] and np.array_equal(bits(got), bits(want)), (s, a, b)
            want, _ = og.run_restart([s], [1.0], 1, C015, n_iter=a + b, init_node=s)
            assert np.array_equal(bits(got), bits(want))
        got, it = og.run_ops(og.constructor_rank(s), [fixed(0), threshold(1e-9, 3000)], C015, seed=s)
        want, iw = og.run(s, C015, threshold=1e-9, max_iter=3000)
        assert it[1] == iw and np.array_equal(bits(got), bits(want))
    nodes = rng.sample(range(og.n), 3)
    w = [0.5, 0.3, 0.2]
    got, _ = og.run_ops(og.n * np.bincount(nodes, w, og.n), [fixed(3), fixed(4)], C015, nodes=nodes, weights=w)
    want, _ = og.run_restart(nodes, w, 2, C015, n_iter=7)
    assert np.array_equal(bits(got), bits(want))
