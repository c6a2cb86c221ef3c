"""Continuing a result on the device (rwr_continue_fixed / rwr_continue_threshold) and writing its rank (rwr_set_rank):
`Model.run(a); run(b)` is `run(a + b)` bit for bit -- seeded, uniform, restart sets, FP64 and FP32, both layouts, with the
sparse prefix forced and off -- a threshold run after a fixed one and a caller-written rank match the resume oracle
(tests/resume_oracle.cpp), rankings of continued results, isolation from the cached iteration graph, the error codes and
the Python Model."""
import ctypes as C
import random
import re

import numpy as np
import pytest

from conftest import C1_SPEC, bits, load_golden
import oracle as O
from resume_oracle import ResumeOracle, fixed, threshold

pytestmark = pytest.mark.gpu

import recommendersystems_b200 as rs
from recommendersystems_b200 import _native as N
from recommendersystems_b200.rwr import run_fixed, run_fixed_restart, run_threshold, run_threshold_restart

from test_gpu_parity import C015, assert_close_fp32, assert_close_fp64, gpu_graph, same_ranking
from test_gpu_frontier import SCALE_C2_NINTH
from test_gpu_restart import UNIT_SPEC, restart_sets, special_nodes

PAIRS = [(0, 1), (0, 7), (1, 1), (1, 5), (2, 3), (5, 15)]
THR = 1e-6


@pytest.fixture(scope="module")
def c1():
    cpu = O.synth_generate(C1_SPEC)
    og = ResumeOracle(cpu)
    gg = rs.Graph.synthetic(C1_SPEC)
    gg.buildGraph()
    return cpu, og, gg


@pytest.fixture(scope="module")
def unit():
    gi = rs.Graph.synthetic(UNIT_SPEC, layout=N.LAYOUT_INDEX)
    gi.buildGraph()
    gv = rs.Graph.synthetic(UNIT_SPEC, layout=N.LAYOUT_VALUED)
    gv.buildGraph()
    return O.synth_generate(UNIT_SPEC), gi, gv


def all_scores(res):
    out = np.stack([res.scores(s) for s in range(res.n_seeds)])
    res.close()
    return out


def seeds_of(cpu, n):
    """a hub, a user, ITEM nodes, a node without links if any, and the uniform restart"""
    return special_nodes(cpu, n) + [-1]


def bound(prec, max_iter):
    """FP32 ranks of a graph this size need not reach a threshold of the FP64 bar: its threshold runs are bounded"""
    return max_iter if prec == rs.FP64 or max_iter > 0 else 200


@pytest.fixture(params=["sparse", "dense"])
def frontier(request, monkeypatch):
    """the sparse prefix forced on (and traced), or off"""
    if request.param == "sparse":
        monkeypatch.setenv("RWR_FRONTIER_BUDGET", "1000000")
        monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
        monkeypatch.delenv("RWR_NO_FRONTIER", raising=False)
    else:
        monkeypatch.setenv("RWR_NO_FRONTIER", "1")
    return request.param


# ------------------------------------------------------------------------------------------ bit identity of continuation
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_fixed_continuation_equals_one_run_of_the_total(c1, prec, frontier):
    cpu, og, gg = c1
    seeds = seeds_of(cpu, og.n)
    for a, b in PAIRS:
        want = all_scores(run_fixed(gg, seeds, C015, a + b, prec))
        r = run_fixed(gg, seeds, C015, a, prec)
        r.continue_fixed(b)
        assert r.info().iterations == a + b
        assert np.array_equal(bits(all_scores(r)), bits(want)), (a, b)
        for s in seeds:                                     # one seed per result: the replayed sparse prefix per slot
            want1 = all_scores(run_fixed(gg, [s], C015, a + b, prec))
            r = run_fixed(gg, [s], C015, a, prec)
            r.continue_fixed(b)
            assert np.array_equal(bits(all_scores(r)), bits(want1)), (s, a, b)
    # chains of continuations
    want = all_scores(run_fixed(gg, seeds, C015, 13, prec))
    r = run_fixed(gg, seeds, C015, 1, prec)
    for b in (1, 1, 3, 0, -2, 7):
        r.continue_fixed(b)
    assert r.info().iterations == 13
    assert np.array_equal(bits(all_scores(r)), bits(want))


def test_the_sparse_prefix_runs_in_continuations(c1, frontier, capfd):
    cpu, og, gg = c1
    if frontier != "sparse":
        pytest.skip("traced with the sparse prefix forced")
    hub = special_nodes(cpu, og.n)[0]
    capfd.readouterr()
    r = run_fixed(gg, [hub], C015, 1)
    r.continue_fixed(5)                                     # replays from the constructor: 2 sparse of 6
    r.continue_fixed(3)                                     # dense from the held rank
    err = capfd.readouterr().err
    got = [(int(a), int(b)) for a, b in re.findall(r"\[rwr frontier\] seed -?\d+: (\d+) of (\d+) iterations sparse", err)]
    assert got == [(1, 1), (2, 6), (0, 3)], got
    want = all_scores(run_fixed(gg, [hub], C015, 9))
    assert np.array_equal(bits(all_scores(r)), bits(want))


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_fixed_continuation_in_both_layouts(unit, prec, frontier):
    cpu, gi, gv = unit
    n = gi.size()
    seeds = seeds_of(cpu, n)
    for gg in (gi, gv):
        for a, b in ((1, 5), (2, 3), (5, 15)):
            want = all_scores(run_fixed(gg, seeds, C015, a + b, prec))
            r = run_fixed(gg, seeds, C015, a, prec)
            r.continue_fixed(b)
            assert np.array_equal(bits(all_scores(r)), bits(want)), (a, b)


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_fixed_continuation_on_a_column_blocked_graph(c1, prec):
    """x_blocks > 1 (the BMODE 1 epilogues): seeded, uniform and restart-set continuations, and a rank written back"""
    cpu, og, _ = c1
    gb = rs.Graph.synthetic(C1_SPEC, x_blocks=4)
    gb.buildGraph()
    assert gb.info().x_blocks > 1
    seeds = seeds_of(cpu, og.n)
    nodes, weights = restart_sets(cpu, og.n, random.Random(6))[1]
    for a, b in ((0, 7), (1, 5), (5, 15)):
        want = all_scores(run_fixed(gb, seeds, C015, a + b, prec))
        r = run_fixed(gb, seeds, C015, a, prec)
        r.continue_fixed(b)
        assert np.array_equal(bits(all_scores(r)), bits(want)), (a, b)
        want = all_scores(run_fixed_restart(gb, nodes, weights, C015, a + b, rs.INIT_RESTART, 0, prec))
        r = run_fixed_restart(gb, nodes, weights, C015, a, rs.INIT_RESTART, 0, prec)
        r.continue_fixed(b)
        assert np.array_equal(bits(all_scores(r)), bits(want)), ("set", a, b)
    for s in seeds:
        x = run_fixed(gb, [s], C015, 5, prec)
        y = run_fixed(gb, [s], C015, 5, prec)
        y.set_rank(0, y.scores(0))
        x.continue_fixed(4)
        y.continue_fixed(4)
        assert np.array_equal(bits(all_scores(x)), bits(all_scores(y))), s
    gb.close()


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_restart_set_continuation_under_every_init(c1, prec):
    cpu, og, gg = c1
    rng = random.Random(5)
    for nodes, weights in restart_sets(cpu, og.n, rng):
        for init in (rs.INIT_UNIFORM, rs.INIT_NODE, rs.INIT_RESTART):
            for a, b in PAIRS:
                want = all_scores(run_fixed_restart(gg, nodes, weights, C015, a + b, init, nodes[0], prec))
                r = run_fixed_restart(gg, nodes, weights, C015, a, init, nodes[0], prec)
                r.continue_fixed(b)
                assert np.array_equal(bits(all_scores(r)), bits(want)), (len(nodes), init, a, b)


def test_scale_c2_ninth_continuation(monkeypatch, capfd):
    """the 22 M-link graph with the default budget of E/64: run(10) + continuation(10) = run(20), sparse prefix traced"""
    monkeypatch.delenv("RWR_NO_FRONTIER", raising=False)
    monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
    gg = rs.Graph.synthetic(SCALE_C2_NINTH)
    gg.buildGraph()
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", str(gg.info().nnz // 64))
    deg = gg.degrees(raw=True)
    seed = int(np.flatnonzero((deg[:SCALE_C2_NINTH["n_users"]] > 10) & (deg[:SCALE_C2_NINTH["n_users"]] < 60))[0])
    capfd.readouterr()
    want = all_scores(run_fixed(gg, [seed], C015, 20))
    r = run_fixed(gg, [seed], C015, 1)
    r.continue_fixed(9)
    r.continue_fixed(10)
    err = capfd.readouterr().err
    assert re.findall(r"iterations sparse", err) and "seed %d: 2 of 20" % seed in err
    assert np.array_equal(bits(all_scores(r)), bits(want))
    gg.close()


# ------------------------------------------------------------------------------------------ threshold continuations
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_threshold_from_the_constructor_state_equals_run_threshold(c1, prec):
    cpu, og, gg = c1
    seeds = seeds_of(cpu, og.n)
    for thr, max_iter in ((THR, 0), (1e-3, 0), (THR, 4), (0.0, 40)):
        max_iter = bound(prec, max_iter)
        want, wi = run_threshold(gg, seeds, C015, thr, max_iter, prec)
        r = run_fixed(gg, seeds, C015, 0, prec)
        it = r.continue_threshold(thr, max_iter)
        assert it.tolist() == wi.tolist()
        assert np.array_equal(bits(all_scores(r)), bits(all_scores(want))), (thr, max_iter)
    nodes, weights = restart_sets(cpu, og.n, random.Random(3))[1]
    w = [x / sum(weights) for x in weights]
    want, wi = run_threshold_restart(gg, nodes, w, C015, THR, bound(prec, 0), rs.INIT_RESTART, 0, prec)
    r = run_fixed_restart(gg, nodes, w, C015, 0, rs.INIT_RESTART, 0, prec)
    assert r.continue_threshold(THR, bound(prec, 0)).tolist() == [wi]
    assert np.array_equal(bits(all_scores(r)), bits(all_scores(want)))


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_threshold_after_a_fixed_run_matches_the_oracle(c1, prec):
    cpu, og, gg = c1
    for s in special_nodes(cpu, og.n):                     # (the oracle's uniform restart is the O(N^2) literal loop)
        for a, thr, max_iter in ((5, THR, 0), (2, 1e-3, 0), (3, THR, 6)):
            max_iter = bound(prec, max_iter)
            want, wi = og.run_ops(og.constructor_rank(s), [fixed(a), threshold(thr, max_iter)], C015, seed=s)
            r = run_fixed(gg, [s], C015, a, prec)
            it = int(r.continue_threshold(thr, max_iter)[0])
            got = all_scores(r)[0]
            if prec == rs.FP64:
                assert it == wi[1], (s, a, thr)
                assert_close_fp64(got, want, f"seed {s} run({a}); run({thr})")
            else:
                assert_close_fp32(got, want, f"seed {s} run({a}); run({thr})")
    # run() after run(int): the default threshold, bounded
    s = special_nodes(cpu, og.n)[0]
    want, wi = og.run_ops(og.constructor_rank(s), [fixed(4), (2, 30, 0.0)], C015, seed=s)
    r = run_fixed(gg, [s], C015, 4, prec)
    it = int(r.continue_threshold(0.0, 30)[0])
    if prec == rs.FP64:
        assert it == wi[1]
        assert_close_fp64(all_scores(r)[0], want, "run(4); run()")
    else:
        assert_close_fp32(all_scores(r)[0], want, "run(4); run() FP32")


# ------------------------------------------------------------------------------------------ written ranks
def written_vectors(rng, n):
    pos = np.array([rng.random() * 2 + 1e-3 for _ in range(n)])
    zeros = pos.copy()
    zeros[rng.sample(range(n), n // 2)] = 0.0
    return [pos, zeros]


def test_written_rank_matches_the_oracle(c1):
    cpu, og, gg = c1
    rng = random.Random(11)
    for s in seeds_of(cpu, og.n):
        for v in written_vectors(rng, og.n):
            want, _ = og.run_ops(v, [fixed(5)], C015, seed=s)
            for prec in (rs.FP64, rs.FP32):
                r = run_fixed(gg, [s], C015, 3, prec)
                r.set_rank(0, v)
                assert r.info().iterations == 0
                r.continue_fixed(5)
                assert r.info().iterations == 5
                got = all_scores(r)[0]
                if prec == rs.FP64:
                    if s >= 0:
                        assert_close_fp64(got, want, f"seed {s} written rank")
                    else:
                        assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
                else:
                    assert_close_fp32(got, want, f"seed {s} written rank FP32")
            if s < 0:
                continue                                    # (the oracle's uniform restart is the O(N^2) literal loop)
            want, wi = og.run_ops(v, [threshold(THR)], C015, seed=s)
            r = run_fixed(gg, [s], C015, 0)
            r.set_rank(0, v)
            assert int(r.continue_threshold(THR)[0]) == wi[0]
            assert_close_fp64(all_scores(r)[0], want, f"seed {s} written rank, threshold")
    nodes, weights = restart_sets(cpu, og.n, rng)[1]
    v = written_vectors(rng, og.n)[0]
    want, _ = og.run_ops(v, [fixed(4)], C015, nodes=nodes, weights=weights)
    r = run_fixed_restart(gg, nodes, weights, C015, 2)
    r.set_rank(0, v)
    r.continue_fixed(4)
    assert_close_fp64(all_scores(r)[0], want, "restart set, written rank")


def test_written_nan_and_inf_poison_every_node(c1):
    cpu, og, gg = c1
    for bad in (np.nan, np.inf):
        v = np.ones(og.n)
        v[17] = bad
        for s in (special_nodes(cpu, og.n)[0], -1):
            want, _ = og.run_ops(v, [fixed(2)], C015, seed=s)
            assert np.isnan(want).all()
            for prec in (rs.FP64, rs.FP32):
                r = run_fixed(gg, [s], C015, 1, prec)
                r.set_rank(0, v)
                r.continue_fixed(2)
                assert np.isnan(all_scores(r)[0]).all(), (bad, s, prec)


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_writing_back_the_held_rank_changes_no_bit(c1, prec, monkeypatch):
    """after a dense last iteration, the S recomputed from the written-back rank is the epilogue's S"""
    monkeypatch.setenv("RWR_NO_FRONTIER", "1")
    cpu, og, gg = c1
    for s in seeds_of(cpu, og.n):
        a = run_fixed(gg, [s], C015, 5, prec)
        b = run_fixed(gg, [s], C015, 5, prec)
        b.set_rank(0, b.scores(0))
        a.continue_fixed(4)
        b.continue_fixed(4)
        assert np.array_equal(bits(all_scores(a)), bits(all_scores(b))), s
    nodes, weights = restart_sets(cpu, og.n, random.Random(2))[0]
    a = run_fixed_restart(gg, nodes, weights, C015, 3, precision=prec)
    b = run_fixed_restart(gg, nodes, weights, C015, 3, precision=prec)
    b.set_rank(0, b.scores(0))
    a.continue_fixed(2)
    b.continue_fixed(2)
    assert np.array_equal(bits(all_scores(a)), bits(all_scores(b)))


def test_warm_start_after_a_hold_out_matches_the_oracle(c1):
    """ranks of the full graph written into a Model on the same input with users held out, then a threshold run"""
    cpu, og, gg = c1
    s = special_nodes(cpu, og.n)[1]
    ranks = all_scores(run_fixed(gg, [s], C015, 30))[0]
    g2 = rs.Graph.synthetic(C1_SPEC)
    types = np.asarray(cpu["node_type"])
    users = [u for u in np.flatnonzero(types == 1)[:200].tolist() if u != s]
    g2.hold_out(users, 5, 0)
    g2.buildGraph()
    og2 = ResumeOracle(g2.export_links())
    want, wi = og2.run_ops(ranks, [threshold(THR)], C015, seed=s)
    r = run_fixed(g2, [s], C015, 0)
    r.set_rank(0, ranks)
    it = int(r.continue_threshold(THR)[0])
    assert it == wi[0]
    assert_close_fp64(all_scores(r)[0], want, "warm start")
    _, cold = run_threshold(g2, [s], C015, THR)
    assert it < int(cold[0])
    g2.close()


# ------------------------------------------------------------------------------------------ rankings
def test_rankings_of_continued_and_written_results(c1):
    cpu, og, gg = c1
    s = special_nodes(cpu, og.n)[1]
    r = run_fixed(gg, [s], C015, 3)
    r.continue_fixed(7)
    want, _ = og.run(s, C015, n_iter=10)
    ids, sc, _ = r.rank_all(0)
    wids, wsc = og.rank_scores(s, want)
    same_ranking(ids, sc, wids, wsc)
    tids, tsc, cnt = r.topk(10)
    same_ranking(tids[0, :cnt[0]], tsc[0, :cnt[0]], wids[:10], wsc[:10])
    v = written_vectors(random.Random(4), og.n)[0]
    r.set_rank(0, v)
    r.continue_fixed(3)
    want, _ = og.run_ops(v, [fixed(3)], C015, seed=s)
    ids, sc, _ = r.rank_all(0)
    wids, wsc = og.rank_scores(s, want)
    same_ranking(ids, sc, wids, wsc)
    r.close()
    nodes, weights = restart_sets(cpu, og.n, random.Random(8))[1]
    r = run_fixed_restart(gg, nodes, weights, C015, 2)
    r.continue_fixed(6)
    want, _ = og.run_restart(nodes, weights, rs.INIT_RESTART, C015, n_iter=8)
    ids, sc, _ = r.rank_all(0)
    wids, wsc = og.rank_scores_set(nodes, want)
    same_ranking(ids, sc, wids, wsc)
    r.close()


# ------------------------------------------------------------------------------------------ isolation
def test_continuations_leave_the_seeded_graph_and_reruns_alone(c1):
    cpu, og, gg = c1
    s = special_nodes(cpu, og.n)[0]

    def seeded():
        r = run_fixed(gg, [s], C015, 20)
        launches = r.info().kernel_launches
        return all_scores(r), launches
    seeded()
    before, l_before = seeded()
    r = run_fixed(gg, [s], C015, 0)
    r.continue_fixed(20)                                    # the same n_iter: would hit the graph's key if it were cached
    r.continue_fixed(3)
    r.set_rank(0, np.ones(og.n))
    r.continue_threshold(THR)
    after, l_after = seeded()
    assert np.array_equal(bits(before), bits(after)) and l_before == l_after
    r.rerun([s], C015, 20)
    assert np.array_equal(bits(all_scores(r)), bits(before))


def test_error_codes(c1, monkeypatch):
    cpu, og, gg = c1
    L = N.lib()
    v = np.ones(og.n)
    pv = v.ctypes.data_as(C.c_void_p)
    it = np.zeros(2, np.int32)
    assert L.rwr_continue_fixed(None, 3) == N.RWR_E_INVALID
    assert L.rwr_continue_threshold(None, THR, 0, it.ctypes.data_as(C.c_void_p)) == N.RWR_E_INVALID
    assert L.rwr_set_rank(None, 0, pv) == N.RWR_E_INVALID
    r = run_fixed(gg, [0, 1], C015, 2)
    assert L.rwr_continue_threshold(r._h, THR, 0, None) == N.RWR_E_INVALID
    assert L.rwr_set_rank(r._h, 0, None) == N.RWR_E_INVALID
    assert L.rwr_set_rank(r._h, -1, pv) == N.RWR_E_INVALID
    assert L.rwr_set_rank(r._h, 2, pv) == N.RWR_E_INVALID
    assert L.rwr_continue_fixed(r._h, 0) == N.RWR_OK and r.info().iterations == 2
    r.close()
    monkeypatch.setenv("RWR_FAKE_COMM", "1")
    try:
        comm = rs.Comm(0, 2, bytes(128), device=0)
    except (rs.RwrError, OSError) as e:
        pytest.skip(f"no communicator on this machine: {e}")
    gp = rs.Graph.synthetic(dict(C1_SPEC, n_users=200, n_items=900, n_like=3000, n_friend=800, n_follow=50, n_mention=40),
                            comm=comm)
    gp.buildGraph()
    assert gp.info().n_ranks == 2
    rp = run_fixed(gp, [1], C015, 2)
    vp = np.ones(gp.size())
    assert L.rwr_continue_fixed(rp._h, 3) == N.RWR_E_UNSUPPORTED
    assert L.rwr_continue_threshold(rp._h, THR, 0, it.ctypes.data_as(C.c_void_p)) == N.RWR_E_UNSUPPORTED
    assert L.rwr_set_rank(rp._h, 0, vp.ctypes.data_as(C.c_void_p)) == N.RWR_E_UNSUPPORTED
    rp.close()
    m = rs.Model(gp, C015, 1)                              # the Python host refuses the write before touching its result
    m.run(2)
    held, before = m._res, m.rank
    with pytest.raises(rs.RwrError):
        m.rank = vp
    assert m._res is held and np.array_equal(bits(m.rank), bits(before))
    m._res.close()
    gp.close()
    comm.close()


# ------------------------------------------------------------------------------------------ Python host
def test_python_model_continues_on_the_device(c1):
    cpu, og, gg = c1
    s = special_nodes(cpu, og.n)[1]
    m = rs.Model(gg, C015, s)
    m.run(3)
    m.run(4)
    assert m._res.info().kernel_launches == 1 + 3 * 4       # k_init_resume and 4 iterations, not 7
    m7 = rs.Model(gg, C015, s)
    m7.run(7)
    assert np.array_equal(bits(m.rank), bits(m7.rank)) and m.nIterations == 7
    m = rs.Model(gg, C015, s)
    m.run(5)
    thr = 1e-9 * og.n
    m.run(thr)
    want, wi = og.run_ops(og.constructor_rank(s), [fixed(5), threshold(thr)], C015, seed=s)
    assert m.nIterations == 5 + wi[1]
    assert_close_fp64(m.rank, want, "run(5); run(thr)")
    # k deliverRanks / updateRanks pairs are run(k)
    m = rs.Model(gg, C015, s)
    for k in range(6):
        m.deliverRanks()
        nxt = m.nextRank.copy()
        m.deliverRanks()                                    # a second call before updateRanks() changes nothing
        assert np.array_equal(bits(m.nextRank), bits(nxt))
        m.updateRanks()
    m6 = rs.Model(gg, C015, s)
    m6.run(6)
    assert np.array_equal(bits(m.rank), bits(m6.rank)) and m.nIterations == 6
    # a checkConvergence loop stops where run(thr) stops
    m = rs.Model(gg, C015, s)
    n = 0
    while True:
        m.deliverRanks()
        n += 1
        if m.checkConvergence(1e-3):
            m.updateRanks()
            break
        m.updateRanks()
    mt = rs.Model(gg, C015, s)
    mt.run(1e-3)
    assert n == mt.nIterations
    assert np.array_equal(bits(m.rank), bits(mt.rank))
    # the rank setter: a warm start
    v = written_vectors(random.Random(9), og.n)[0]
    m = rs.Model(gg, C015, s)
    m.rank = v
    m.run(THR)
    want, wi = og.run_ops(v, [threshold(THR)], C015, seed=s)
    assert m.nIterations == wi[0]
    assert_close_fp64(m.rank, want, "rank setter")


CPP_SEQUENCES = r'''
// run(3); run(4) | run(5); run(thr) | rank = v; run(thr) | run(2); rank = v; run(3) through RWRBased.hpp: ranks as hex
#include <cstdio>
#include <cstdlib>
#include "RWRBased.hpp"
using namespace Recommenders::RWRBased;

static void print(const char* what, const Model& m) {
    std::printf("%s %d", what, m.nIterations);
    for (double x : m.rank) std::printf(" %a", x);
    std::printf("\n");
}

int main(int argc, char** argv) {
    std::FILE* f = std::fopen(argv[1], "r");
    const int seed = std::atoi(argv[2]);
    const double c = std::strtod(argv[3], nullptr), thr = std::strtod(argv[4], nullptr);
    Dictionary<int, Node> nodes;
    Dictionary<int, List<ForwardLink>> edges;
    int n = 0;
    long long links = 0;
    if (std::fscanf(f, "%d", &n) != 1) return 2;
    for (int i = 0; i < n; i++) {
        long long id;
        int type;
        if (std::fscanf(f, "%lld %d", &id, &type) != 2) return 2;
        nodes.Add(i, Node(id, (NodeType)type));
    }
    if (std::fscanf(f, "%lld", &links) != 1) return 2;
    for (long long k = 0; k < links; k++) {
        int s, d, t;
        double w;
        if (std::fscanf(f, "%d %d %d %la", &s, &d, &t, &w) != 4) return 2;
        if (!edges.ContainsKey(s)) edges.Add(s, List<ForwardLink>());
        edges[s].Add(ForwardLink(d, (EdgeType)t, w));
    }
    std::fclose(f);
    Graph graph(nodes, edges);
    graph.buildGraph();
    std::vector<double> v((size_t)n);
    for (int i = 0; i < n; i++) v[(size_t)i] = 1.0 + (i % 7) * 0.25;
    try {
        Model a(graph, c, seed);
        a.run(3);
        a.run(4);
        print("fixed", a);
        Model b(graph, c, seed);
        b.run(5);
        b.run(thr);
        print("threshold", b);
        Model w(graph, c, seed);
        w.rank = v;
        w.run(thr);
        print("warm", w);
        Model x(graph, c, seed);
        x.run(2);
        x.rank = v;
        x.run(3);
        Model moved(std::move(x));
        print("written", moved);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    return 0;
}
'''


def test_cpp_host_equals_the_python_host(c1, tmp_path):
    """the same sequences through cpp/RWRBased.hpp and through the Python Model: the same bits"""
    import os
    import subprocess
    from conftest import ROOT
    from test_cpp_host import write_graph
    cpu, og, gg = c1
    pkg = os.path.join(ROOT, "recommendersystems_b200")
    src = tmp_path / "resume_sequences.cpp"
    src.write_text(CPP_SEQUENCES)
    exe = str(tmp_path / "resume_sequences")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-I", os.path.join(pkg, "cpp"),
                           "-o", exe, str(src), "-L", pkg, "-lrwr_b200", "-Wl,-rpath," + pkg])
    graph_file = write_graph(str(tmp_path / "c1.txt"), cpu)
    s = special_nodes(cpu, og.n)[1]
    thr = 1e-9 * og.n
    p = subprocess.run([exe, graph_file, str(s), repr(C015), repr(thr)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    got = {}
    for line in p.stdout.splitlines():
        what, iters, *vals = line.split()
        got[what] = (int(iters), np.array([float.fromhex(x) for x in vals]))
    v = np.array([1.0 + (i % 7) * 0.25 for i in range(og.n)])
    a = rs.Model(gg, C015, s); a.run(3); a.run(4)
    b = rs.Model(gg, C015, s); b.run(5); b.run(thr)
    w = rs.Model(gg, C015, s); w.rank = v; w.run(thr)
    x = rs.Model(gg, C015, s); x.run(2); x.rank = v; x.run(3)
    for what, m in (("fixed", a), ("threshold", b), ("warm", w), ("written", x)):
        assert got[what][0] == m.nIterations, what
        assert np.array_equal(bits(got[what][1]), bits(m.rank)), what
