"""Restart sets on the device (rwr_run_fixed_restart / rwr_run_threshold_restart): `Model.restart` overwritten with a
weighted node set.  Bit-identity with the seeded and uniform paths where the restart vector is theirs, the oracle's
restart-set model elsewhere (FP64, FP32, thresholds, NaN / Inf graphs, rankings under the union exclusion, both layouts,
column blocking), and isolation from the seeded path of the same handle."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import C1_SPEC, bits, load_golden
from random_graphs import random_flat
import oracle as O
from restart_oracle import RestartOracle

pytestmark = pytest.mark.gpu

import recommendersystems_b200 as rs
from recommendersystems_b200 import _native as N
from recommendersystems_b200.rwr import run_fixed, run_fixed_restart, run_threshold, run_threshold_restart

from test_gpu_parity import C015, assert_close_fp32, assert_close_fp64, gpu_graph, same_ranking

INITS = [rs.INIT_UNIFORM, rs.INIT_NODE, rs.INIT_RESTART]
UNIT_SPEC = dict(C1_SPEC, n_mention=0)              # one weight per row: builds in both layouts


def scores(res):
    s = res.scores(0)
    res.close()
    return s


@pytest.fixture(scope="module")
def c1():
    cpu = O.synth_generate(C1_SPEC)
    og = RestartOracle(cpu)
    gg = rs.Graph.synthetic(C1_SPEC)
    gg.buildGraph()
    return cpu, og, gg


@pytest.fixture(scope="module")
def unit():
    """the C1 graph without MENTION links, built in the index-only and the valued layout"""
    cpu = O.synth_generate(UNIT_SPEC)
    og = RestartOracle(cpu)
    gi = rs.Graph.synthetic(UNIT_SPEC, layout=N.LAYOUT_INDEX)
    gi.buildGraph()
    gv = rs.Graph.synthetic(UNIT_SPEC, layout=N.LAYOUT_VALUED)
    gv.buildGraph()
    assert gi.info().layout == N.LAYOUT_INDEX and gv.info().layout == N.LAYOUT_VALUED
    return cpu, og, gi, gv


def special_nodes(cpu, n):
    """the biggest hub, a dangling row, a node without raw links if any, users and ITEM nodes"""
    rp_deg = np.bincount(np.asarray(cpu["src"], np.int64), minlength=n)
    types = np.asarray(cpu["node_type"])
    items = np.flatnonzero(types == 2)
    users = np.flatnonzero(types == 1)
    hub = int(np.argmax(rp_deg))
    nolinks = np.flatnonzero(rp_deg == 0)
    out = [hub, int(users[1]), int(items[7]), int(items[len(items) // 2])]
    if len(nolinks):
        out.append(int(nolinks[0]))
    return list(dict.fromkeys(out))


def restart_sets(cpu, n, rng):
    """sets of 2, 17 and 1000 nodes with hubs, dangling rows and ITEM nodes; weights not normalised"""
    sp = special_nodes(cpu, n)
    rest = [v for v in rng.sample(range(n), 1100) if v not in sp]
    s2 = sp[:2]
    s17 = (sp + rest)[:17]
    s1000 = (sp + rest)[:1000]
    w = lambda k: [rng.choice([1.0, 0.5, 2.0, 0.125, rng.random() * 3]) for _ in range(k)]
    return [(s2, w(2)), (s17, w(17)), (s1000, w(1000))]


# ------------------------------------------------------------------------------------------ bit-identity with existing paths
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_one_hot_with_init_node_equals_the_seeded_run_in_both_layouts(unit, prec):
    cpu, og, gi, gv = unit
    for gg in (gi, gv):
        for s in special_nodes(cpu, og.n)[:4]:
            for n_iter in (1, 2, 7, 20):
                a = scores(run_fixed(gg, [s], C015, n_iter, prec))
                b = scores(run_fixed_restart(gg, [s], [1.0], C015, n_iter, rs.INIT_NODE, s, prec))
                assert np.array_equal(bits(a), bits(b)), (s, n_iter, prec)


def test_one_hot_threshold_run_equals_the_seeded_run(unit):
    cpu, og, gi, gv = unit
    for gg in (gi, gv):
        for s in special_nodes(cpu, og.n)[:3]:
            for thr in (1e-3 * og.n, 1e-9 * og.n):
                ra, ia = run_threshold(gg, [s], C015, thr)
                rb, ib = run_threshold_restart(gg, [s], [1.0], C015, thr, 0, rs.INIT_NODE, s)
                assert int(ia[0]) == ib, (s, thr)
                assert np.array_equal(bits(scores(ra)), bits(scores(rb))), (s, thr)


def test_all_nodes_at_one_over_n_equal_the_uniform_constructor(c1):
    cpu, og, gg = c1
    n = og.n
    for n_iter in (1, 5, 20):
        a = scores(run_fixed(gg, [-1], C015, n_iter))
        b = scores(run_fixed_restart(gg, np.arange(n), np.full(n, 1.0 / n), C015, n_iter, rs.INIT_UNIFORM))
        assert np.array_equal(bits(a), bits(b)), n_iter


# ------------------------------------------------------------------------------------------ against the oracle
def check_against_oracle(og, gg, nodes, weights, init, init_node, iters=(1, 2, 20), fp32=True, what=""):
    for it in iters:
        want, _ = og.run_restart(nodes, weights, init, C015, n_iter=it, init_node=init_node)
        got = scores(run_fixed_restart(gg, nodes, weights, C015, it, init, init_node))
        assert_close_fp64(got, want, f"{what} init {init} iter {it}")
    if fp32:
        # q is not normalised: 20 iterations of a set whose weights sum to ~1000 grow the ranks past 1e38, beyond FP32
        w = np.asarray(weights) / np.sum(weights)
        want, _ = og.run_restart(nodes, w, init, C015, n_iter=20, init_node=init_node)
        got = scores(run_fixed_restart(gg, nodes, w, C015, 20, init, init_node, rs.FP32))
        assert_close_fp32(got, want, f"{what} fp32 init {init}")


def test_c1_sets_against_the_oracle(c1):
    cpu, og, gg = c1
    rng = random.Random(41)
    for nodes, weights in restart_sets(cpu, og.n, rng):
        for init in INITS:
            check_against_oracle(og, gg, nodes, weights, init, nodes[0], what=f"C1 m={len(nodes)}")


def test_c1_threshold_iteration_counts(c1):
    cpu, og, gg = c1
    rng = random.Random(42)
    for nodes, weights in restart_sets(cpu, og.n, rng)[:2]:
        w = np.asarray(weights) / np.sum(weights)        # mass N is kept: the runs converge
        for init in INITS:
            for thr in (1e-3, 1e-6, 1e-9, 1e-12):
                want, want_it = og.run_restart(nodes, w, init, C015, threshold=thr * og.n, init_node=nodes[0], max_iter=5000)
                res, it = run_threshold_restart(gg, nodes, w, C015, thr * og.n, 0, init, nodes[0])
                assert it == want_it, (len(nodes), init, thr, it, want_it)
                assert_close_fp64(scores(res), want, f"threshold m={len(nodes)} init {init} thr {thr}")


def test_c1_rankings_under_the_union_exclusion(c1):
    cpu, og, gg = c1
    rng = random.Random(43)
    for nodes, weights in restart_sets(cpu, og.n, rng):
        want, _ = og.run_restart(nodes, weights, rs.INIT_RESTART, C015, n_iter=20)
        wids, wsc = og.rank_scores_set(nodes, want)
        res = run_fixed_restart(gg, nodes, weights, C015, 20)
        ids, sc, cnt = res.rank_all(0)
        assert cnt == len(wids)
        same_ranking(ids, sc, wids, wsc)
        for k in (10, 40):                                    # k <= 16: block scan; k > 16: the full-ranking path
            tids, tsc, tcnt = res.topk(k)
            same_ranking(tids[0, :tcnt[0]], tsc[0, :tcnt[0]], wids[:k], wsc[:k])
        res.close()


def test_index_layout_sets_against_the_oracle(unit):
    cpu, og, gi, gv = unit
    rng = random.Random(44)
    for nodes, weights in restart_sets(cpu, og.n, rng)[:2]:
        for init in INITS:
            check_against_oracle(og, gi, nodes, weights, init, nodes[-1], iters=(1, 20), what="index")
            check_against_oracle(og, gv, nodes, weights, init, nodes[-1], iters=(20,), fp32=False, what="valued")


def test_column_blocked_graph_against_the_oracle(c1):
    cpu, og, _ = c1
    gb = rs.Graph.synthetic(C1_SPEC, x_blocks=4)
    gb.buildGraph()
    assert gb.info().x_blocks > 1
    rng = random.Random(45)
    for nodes, weights in restart_sets(cpu, og.n, rng)[:2]:
        for init in INITS:
            check_against_oracle(og, gb, nodes, weights, init, nodes[0], iters=(1, 20), what="x_blocks")
        w = np.asarray(weights) / np.sum(weights)
        _, want_it = og.run_restart(nodes, w, rs.INIT_RESTART, C015, threshold=1e-6 * og.n, max_iter=5000)
        _, it = run_threshold_restart(gb, nodes, w, C015, 1e-6 * og.n)
        assert it == want_it
    gb.close()


@pytest.mark.parametrize("case", range(4))
def test_nan_and_inf_graphs_give_the_oracles_nan_set(case):
    rng = random.Random(20261000 + case)
    f = random_flat(rng, rng.randrange(3, 12), rng.randrange(5, 60), rng.randrange(0, 4), rng.randrange(20, 400),
                    zero_rows=1, nan_rows=1)
    gg, og = gpu_graph(f), RestartOracle(f)
    n = og.n
    poisoned = 0
    for m in (1, 2, min(17, n)):
        nodes = rng.sample(range(n), m)
        weights = [rng.choice([1.0, 0.5, 0.0, 2.0]) for _ in range(m)]
        for init in INITS:
            for it in (1, 2, 3, 8):
                want, _ = og.run_restart(nodes, weights, init, C015, n_iter=it, init_node=nodes[0])
                got = scores(run_fixed_restart(gg, nodes, weights, C015, it, init, nodes[0]))
                assert np.array_equal(np.isnan(got), np.isnan(want)), (m, init, it)
                assert np.array_equal(np.isinf(got), np.isinf(want)), (m, init, it)
                ok = np.isfinite(want)
                assert_close_fp64(got[ok], want[ok], f"nan graph m={m} init {init} iter {it}")
                poisoned += int(np.isnan(want).all())
    assert poisoned > 0
    gg.close()


def test_golden_graphs_against_the_oracle():
    for name in ("kat_8c", "small_a", "small_b"):
        inp = load_golden(name)["input"]
        gg, og = gpu_graph(inp), RestartOracle(inp)
        n = og.n
        for nodes, weights in ([0], [1.0]), ([0, n - 1], [0.75, 0.25]), (list(range(n)), [1.0] * n):
            for init in INITS:
                check_against_oracle(og, gg, nodes, weights, init, nodes[-1], iters=(1, 2, 10), fp32=False, what=name)
        gg.close()


# ------------------------------------------------------------------------------------------ isolation
def test_reruns_are_bit_identical_and_the_seeded_path_is_untouched(c1, monkeypatch):
    cpu, og, gg = c1
    rng = random.Random(46)
    seed = special_nodes(cpu, og.n)[1]
    sets = restart_sets(cpu, og.n, rng)

    def seeded():
        r = run_fixed(gg, [seed], C015, 20)
        launches = r.info().kernel_launches
        return scores(r), launches
    seeded()                                               # first run of this key: kernel by kernel
    before, l_before = seeded()                            # second: the captured iteration graph
    for prec in (rs.FP64, rs.FP32):
        for nodes, weights in sets:
            a = scores(run_fixed_restart(gg, nodes, weights, C015, 20, rs.INIT_RESTART, 0, prec))
            b = scores(run_fixed_restart(gg, nodes, weights, C015, 20, rs.INIT_RESTART, 0, prec))
            assert np.array_equal(bits(a), bits(b))
            ra, ia = run_threshold_restart(gg, nodes, weights, C015, 1e-6 * og.n, 50, rs.INIT_UNIFORM, 0, prec)
            rb, ib = run_threshold_restart(gg, nodes, weights, C015, 1e-6 * og.n, 50, rs.INIT_UNIFORM, 0, prec)
            assert ia == ib and np.array_equal(bits(scores(ra)), bits(scores(rb)))
    after, l_after = seeded()
    assert np.array_equal(bits(before), bits(after)) and l_before == l_after


def test_restart_sets_never_go_sparse(c1, monkeypatch, capfd):
    import re
    cpu, og, gg = c1
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", str(1 << 20))
    monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
    seed = special_nodes(cpu, og.n)[1]
    capfd.readouterr()
    scores(run_fixed(gg, [seed], C015, 5))
    scores(run_fixed_restart(gg, [seed], [1.0], C015, 5, rs.INIT_NODE, seed))
    scores(run_fixed_restart(gg, special_nodes(cpu, og.n), [1.0] * len(special_nodes(cpu, og.n)), C015, 5))
    err = capfd.readouterr().err
    seeded = [int(x) for x in re.findall(r"\[rwr frontier\] seed -?\d+: (\d+) of \d+ iterations sparse", err)]
    sets = [int(x) for x in re.findall(r"\[rwr frontier\] restart set of \d+ nodes: (\d+) of \d+ iterations sparse", err)]
    assert seeded and seeded[0] > 0                        # the trace works: the seeded run went sparse
    assert sets == [0, 0]


def test_validation_codes(c1):
    cpu, og, gg = c1
    L = N.lib()
    n = og.n
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    out = C.c_void_p()
    it = np.zeros(1, np.int32)

    def fixed(nodes, weights, m=None, init=rs.INIT_RESTART, init_node=0):
        nd = None if nodes is None else np.ascontiguousarray(nodes, np.int32)
        w = None if weights is None else np.ascontiguousarray(weights, np.float64)
        m = (len(nd) if nd is not None else 1) if m is None else m
        rc = L.rwr_run_fixed_restart(gg._h, None if nd is None else p(nd), None if w is None else p(w), m, init, init_node,
                                     C015, 5, N.FP64, C.byref(out))
        if rc == N.RWR_OK:
            L.rwr_result_destroy(out)
        rt = L.rwr_run_threshold_restart(gg._h, None if nd is None else p(nd), None if w is None else p(w), m, init, init_node,
                                         C015, 1e-3, 10, N.FP64, p(it), C.byref(out))
        assert rc == rt, (rc, rt)
        return rc
    assert fixed(None, [1.0]) == N.RWR_E_INVALID
    assert fixed([1], None) == N.RWR_E_INVALID
    assert fixed([1], [1.0], m=0) == N.RWR_E_INVALID
    assert fixed([1, 2, 1], [1.0, 1.0, 1.0]) == N.RWR_E_INVALID            # duplicate
    assert fixed([1, 2], [1.0, np.nan]) == N.RWR_E_INVALID
    assert fixed([1, 2], [1.0, np.inf]) == N.RWR_E_INVALID
    assert fixed([1, 2], [1.0, -0.5]) == N.RWR_E_INVALID
    assert fixed([1], [1.0], init=3) == N.RWR_E_INVALID
    assert fixed([1, n], [1.0, 1.0]) == N.RWR_E_BADSEED
    assert fixed([-1], [1.0]) == N.RWR_E_BADSEED
    assert fixed([1], [1.0], init=rs.INIT_NODE, init_node=n) == N.RWR_E_BADSEED
    assert fixed([1], [1.0], init=rs.INIT_NODE, init_node=-1) == N.RWR_E_BADSEED
    assert fixed([1], [1.0], init=rs.INIT_UNIFORM, init_node=-1) == N.RWR_OK            # init_node is read for NODE only
    L.rwr_result_destroy(out)
    res = run_fixed_restart(gg, [1, 2], [1.0, 1.0], C015, 5)
    s = np.array([1], np.int32)
    assert L.rwr_rerun_fixed(res._h, p(s), C015, 5) == N.RWR_E_INVALID
    res.close()


def test_partitioned_handle_is_refused(monkeypatch):
    """A slice of a row-partitioned graph (here the one-GPU RWR_FAKE_COMM slice of two ranks) refuses restart sets."""
    monkeypatch.setenv("RWR_FAKE_COMM", "1")
    try:
        comm = rs.Comm(0, 2, bytes(128), device=0)
    except (rs.RwrError, OSError) as e:
        pytest.skip(f"no communicator on this machine: {e}")
    gp = rs.Graph.synthetic(dict(C1_SPEC, n_users=200, n_items=900, n_like=3000, n_friend=800, n_follow=50, n_mention=40),
                            comm=comm)
    gp.buildGraph()
    assert gp.info().n_ranks == 2
    L = N.lib()
    nd = np.array([1], np.int32)
    w = np.array([1.0])
    out = C.c_void_p()
    rc = L.rwr_run_fixed_restart(gp._h, nd.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), 1, rs.INIT_RESTART, 0,
                                 C015, 5, N.FP64, C.byref(out))
    gp.close()
    comm.close()
    assert rc == N.RWR_E_UNSUPPORTED


# ------------------------------------------------------------------------------------------ Python host surface
def test_model_restart_setter_and_recommendation_for_set(c1):
    cpu, og, gg = c1
    n = og.n
    sp = special_nodes(cpu, og.n)
    q = np.zeros(n)
    q[sp] = [1.0, 0.5, 0.25, 2.0, 1.5][:len(sp)]
    nodes = np.flatnonzero(q)
    for target in (None, sp[1]):
        m = rs.Model(gg, C015) if target is None else rs.Model(gg, C015, target)
        before = m.restart.copy()
        m.restart = q
        assert np.array_equal(m.restart, q)
        m.run(12)
        init = rs.INIT_UNIFORM if target is None else rs.INIT_NODE
        want, _ = og.run_restart(nodes, q[nodes], init, C015, n_iter=12, init_node=0 if target is None else target)
        assert_close_fp64(m.rank, want, f"Model.restart setter, target {target}")
        m2 = rs.Model(gg, C015) if target is None else rs.Model(gg, C015, target)
        m2.restart = before                                # the constructor's vector: today's path
        m2.run(12)
        m3 = rs.Model(gg, C015) if target is None else rs.Model(gg, C015, target)
        m3.run(12)
        assert np.array_equal(bits(m2.rank), bits(m3.rank))
        qn = q / q.sum()
        m4 = rs.Model(gg, C015) if target is None else rs.Model(gg, C015, target)
        m4.restart = qn
        m4.run(1e-6 * n)
        _, want_it = og.run_restart(nodes, qn[nodes], init, C015, threshold=1e-6 * n, init_node=0 if target is None else target,
                                    max_iter=5000)
        assert m4.nIterations == want_it
    rec = rs.Recommender(gg)
    weights = q[nodes]
    want, _ = og.run_restart(nodes, weights, rs.INIT_RESTART, C015, n_iter=20)
    wids, wsc = og.rank_scores_set(nodes, want)
    full = rec.RecommendationForSet(nodes.tolist(), weights.tolist(), 0.15, 20)
    same_ranking([p[0] for p in full], [p[1] for p in full], wids, wsc)
    top = rec.RecommendationForSet(nodes.tolist(), weights.tolist(), 0.15, 20, 10)
    same_ranking([p[0] for p in top], [p[1] for p in top], wids[:10], wsc[:10])
