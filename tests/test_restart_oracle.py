"""CPU tests of restart sets (`Model.restart` overwritten with a weighted node set): the restart-set oracle's collapsed form
(tests/restart_oracle.cpp) against its literal O(N^2) loops and against the pure-Python restatement (oracle/rwr_literal.py),
the one-hot case against the seeded CPU oracle, the union exclusion of the ranking helper, and the argument checks of the
new entry points that need no GPU."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import C1_SPEC, bits
from random_graphs import random_flat
import oracle as O
import rwr_literal as R
from restart_oracle import RestartOracle

from recommendersystems_b200 import _native as N

INIT_UNIFORM, INIT_NODE, INIT_RESTART = 0, 1, 2
C015 = O.widen_float(0.15)


def oracle_of(flat):
    return RestartOracle(flat)


def literal_of(flat):
    pg = R.graph_from_flat(flat["node_id"], flat["node_type"], flat["src"], flat["dst"], flat["etype"], flat["w"])
    pg.buildGraph()
    return pg


def python_model(pg, n, nodes, weights, init, init_node, c):
    """rwr_literal's Model with its public `restart` assigned, from the initial rank of `init`"""
    m = R.Model(pg, c, init_node) if init == INIT_NODE else R.Model(pg, c)
    q = [0.0] * n
    for v, w in zip(nodes, weights):
        q[v] = float(w)
    m.restart = q
    if init == INIT_RESTART:
        m.rank = [float(n) * x for x in q]
    return m


def same(a, b):
    """bit for bit, except that any NaN equals any NaN (the payload of a NaN differs between C++ and Python arithmetic)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(a[~na]), bits(b[~nb]))


def random_set(rng, n, m):
    nodes = rng.sample(range(n), m)
    weights = [rng.choice([1.0, 0.5, 0.0, 3.25, rng.random() * 2]) for _ in range(m)]
    return nodes, weights


GRAPH_SEEDS = [11, 12, 13, 14]


@pytest.mark.parametrize("gseed", GRAPH_SEEDS)
def test_collapsed_equals_literal_and_python_on_random_graphs(gseed):
    """Dangling rows, multi-edges, fractional weights and (for odd seeds) NaN / Inf rows: the sparse collapsed form equals
    the literal loops bit for bit under every init, for several iteration counts and thresholds; rwr_literal agrees."""
    rng = random.Random(gseed)
    poison = gseed % 2 == 1
    flat = random_flat(rng, 8, 20, 3, 90, zero_rows=1 if poison else 0, nan_rows=1 if poison else 0)
    og, pg = oracle_of(flat), literal_of(flat)
    n = og.n
    for m in (1, 2, 5, n):
        nodes, weights = random_set(rng, n, m)
        for init in (INIT_UNIFORM, INIT_NODE, INIT_RESTART):
            init_node = rng.randrange(n)
            for n_iter in (0, 1, 3, 7):
                a, _ = og.run_restart(nodes, weights, init, C015, n_iter=n_iter, init_node=init_node, literal=True)
                b, _ = og.run_restart(nodes, weights, init, C015, n_iter=n_iter, init_node=init_node, literal=False)
                assert np.array_equal(bits(a), bits(b)), (m, init, n_iter)
                pm = python_model(pg, n, nodes, weights, init, init_node, C015)
                pm.run(n_iter)
                assert same(a, pm.rank), (m, init, n_iter, "python")
            if poison:
                continue                                           # NaN ranks never converge: no threshold runs
            # q is not normalised: a set whose weights sum to more than 1 gains mass every iteration and never converges, so
            # the threshold runs take the weights scaled to a sum of 1
            total = sum(weights)
            weights = [w / total for w in weights] if total > 0 else weights
            for thr in (1e-3, 1e-6, 1e-9):
                a, ia = og.run_restart(nodes, weights, init, C015, threshold=thr, init_node=init_node, literal=True, max_iter=2000)
                b, ib = og.run_restart(nodes, weights, init, C015, threshold=thr, init_node=init_node, literal=False, max_iter=2000)
                assert ia == ib and np.array_equal(bits(a), bits(b)), (m, init, thr)
                pm = python_model(pg, n, nodes, weights, init, init_node, C015)
                pm.run(thr)
                assert pm.nDeliver == ia and same(a, pm.rank)


def test_poisoned_graph_spreads_nan_like_the_literal_loops():
    """A row whose weights sum to 0 makes its rank NaN: every entry of the next vector is NaN in the reference, members
    and non-members alike, and the collapsed form reproduces that."""
    rng = random.Random(5)
    flat = random_flat(rng, 6, 12, 2, 60, zero_rows=2, nan_rows=1)
    og = oracle_of(flat)
    n = og.n
    nodes, weights = random_set(rng, n, 3)
    a, _ = og.run_restart(nodes, weights, INIT_UNIFORM, C015, n_iter=4, literal=True)
    b, _ = og.run_restart(nodes, weights, INIT_UNIFORM, C015, n_iter=4, literal=False)
    assert np.isnan(a).any() and np.array_equal(bits(a), bits(b))


def test_c1_collapsed_equals_literal():
    """The C1-shaped synthetic graph: a set with its biggest hub, a dangling row and ITEM nodes, three inits."""
    s = O.synth_generate(C1_SPEC)
    og = RestartOracle(s)
    n = og.n
    rp, _, _ = og.csr()
    deg = np.diff(rp)
    items = np.flatnonzero(np.asarray(s["node_type"]) == 2)
    nodes = [int(np.argmax(deg)), int(np.flatnonzero(deg == 0)[0]), int(items[3]), int(items[500])]
    weights = [1.0, 0.25, 2.5, 0.125]
    for init in (INIT_UNIFORM, INIT_NODE, INIT_RESTART):
        a, _ = og.run_restart(nodes, weights, init, C015, n_iter=2, init_node=nodes[0], literal=True)
        b, _ = og.run_restart(nodes, weights, init, C015, n_iter=2, init_node=nodes[0], literal=False)
        assert np.array_equal(bits(a), bits(b)), init
        assert np.all(a >= 0.0)


@pytest.mark.parametrize("gseed", [21, 22])
def test_one_hot_with_init_node_is_the_seeded_run(gseed):
    """{s: 1.0} with init NODE(s) is `new Model(graph, c, s)` with its own restart vector: the seeded oracle run, bit for bit."""
    rng = random.Random(gseed)
    flat = random_flat(rng, 8, 20, 3, 90, zero_rows=gseed % 2, nan_rows=0)
    og = oracle_of(flat)
    for s in rng.sample(range(og.n), 6):
        for n_iter in (1, 2, 9):
            a, _ = og.run(s, C015, n_iter=n_iter)
            for init in (INIT_NODE, INIT_RESTART):                 # fl(N * 1.0) == N: RESTART starts from the same rank
                b, _ = og.run_restart([s], [1.0], init, C015, n_iter=n_iter, init_node=s)
                assert np.array_equal(bits(a), bits(b)), (s, n_iter, init)
        if gseed % 2 == 0:
            a, ia = og.run(s, C015, threshold=1e-9, max_iter=2000)
            b, ib = og.run_restart([s], [1.0], INIT_NODE, C015, threshold=1e-9, init_node=s, max_iter=2000)
            assert ia == ib and np.array_equal(bits(a), bits(b))


def test_uniform_set_is_the_uniform_constructor():
    """Every node at 1/N with init UNIFORM restates `new Model(graph, c)`: the literal loops of both agree bit for bit."""
    rng = random.Random(3)
    flat = random_flat(rng, 5, 10, 2, 40)
    og = oracle_of(flat)
    n = og.n
    a, _ = og.run(-1, C015, n_iter=5, literal=True)
    b, _ = og.run_restart(list(range(n)), [1.0 / n] * n, INIT_UNIFORM, C015, n_iter=5, literal=True)
    assert np.array_equal(bits(a), bits(b))


def test_set_ranking_excludes_the_union_of_like_targets():
    rng = random.Random(9)
    flat = random_flat(rng, 8, 25, 2, 120)
    og = oracle_of(flat)
    n = og.n
    src, dst, et = (np.asarray(flat[k]) for k in ("src", "dst", "etype"))
    no_links = [v for v in range(n) if not np.any(src == v)]
    nodes = [int(src[0]), int(src[-1])] + no_links[:1]
    rank, _ = og.run_restart(nodes, [1.0] * len(nodes), INIT_RESTART, C015, n_iter=5)
    ids, sc = og.rank_scores_set(nodes, rank)
    liked = {int(d) for s, d, t in zip(src, dst, et) if int(s) in nodes and t == R.LIKE}
    types, node_id = np.asarray(flat["node_type"]), np.asarray(flat["node_id"])
    want = [(int(node_id[i]), rank[i]) for i in range(n) if types[i] == R.ITEM and i not in liked]
    want.sort(key=lambda p: (-p[1], -p[0]))
    assert ids.tolist() == [p[0] for p in want] and np.array_equal(bits(sc), bits(np.array([p[1] for p in want])))
    # one listed node: the seeded ranking helper's exclusion
    s = int(src[0])
    assert np.array_equal(og.rank_scores_set([s], rank)[0], og.rank_scores(s, rank)[0])


def test_entry_points_reject_a_null_graph_without_a_gpu():
    L = N.lib()
    nodes = np.array([0, 1], np.int32)
    w = np.array([1.0, 0.5])
    out = C.c_void_p()
    it = np.zeros(1, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.rwr_run_fixed_restart(None, p(nodes), p(w), 2, N.INIT_RESTART, 0, 0.15, 10, N.FP64, C.byref(out)) == N.RWR_E_INVALID
    assert not out.value
    assert L.rwr_run_threshold_restart(None, p(nodes), p(w), 2, N.INIT_RESTART, 0, 0.15, 1e-6, 0, N.FP64, p(it),
                                       C.byref(out)) == N.RWR_E_INVALID
    assert L.rwr_run_fixed_restart(None, p(nodes), p(w), 2, N.INIT_RESTART, 0, 0.15, 10, N.FP64, None) == N.RWR_E_INVALID
