"""The sparse prefix of a single-seed run (frontier.cu): the first iterations pushed from the seed's frontier instead of
streamed over the whole matrix.  RWR_FRONTIER_BUDGET forces the path on graphs below its size floor (2^25 links); RWR_NO_FRONTIER=1
gives the dense run of the same seed for comparison; RWR_FRONTIER_TRACE=1 makes every run report on stderr how many of
its iterations the frontier kernels did, so the tests see that the sparse path really ran."""
import re

import numpy as np
import pytest

from conftest import bits, load_golden

pytestmark = pytest.mark.gpu

import recommendersystems_b200 as rs
from recommendersystems_b200 import _native as N
from recommendersystems_b200.rwr import run_fixed

from test_gpu_parity import C015, assert_close_fp32, assert_close_fp64, gpu_graph, oracle_graph

CASES = ["kat_8c", "small_a", "small_b"]          # non-uniform row weights: built with the valued layout
SPARSE_ITERS = 2                                  # FR_ITERS of frontier.h
SCALE_C2_NINTH = dict(seed=11, n_users=120_000, n_items=1_100_000, n_third=0, authorship_per_mille=1000, n_like=7_800_000,
                      n_friend=2_200_000, n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1, p1_byte=61)


def uniform6():
    """0 -> {1, 2} (both dangling), 3 dangling, 4 -> 0, 5 -> {4, 0}: one weight per row, so both layouts build"""
    n = 6
    src = np.array([0, 0, 4, 5, 5], np.int32)
    dst = np.array([1, 2, 0, 4, 0], np.int32)
    return dict(node_id=np.arange(n, dtype=np.int64) + 100, node_type=np.array([1, 2, 2, 1, 1, 1], np.int32),
                src=src, dst=dst, etype=np.full(len(src), 2, np.int32), w=np.ones(len(src)))


def traced(capfd, fn):
    """(result of fn(), sparse iterations of the runs fn made, as RWR_FRONTIER_TRACE reports them)"""
    capfd.readouterr()
    out = fn()
    err = capfd.readouterr().err
    return out, [int(m) for m in re.findall(r"\[rwr frontier\] seed -?\d+: (\d+) of \d+ iterations sparse", err)]


def run(gg, seed, n_iter, prec=rs.FP64, dense=False, monkeypatch=None, capfd=None, sparse=None):
    """scores of one fixed-count run; with capfd, asserts that `sparse` of its iterations ran on the frontier kernels"""
    if dense:
        monkeypatch.setenv("RWR_NO_FRONTIER", "1")

    def go():
        r = run_fixed(gg, [seed], C015, n_iter, prec)
        s = r.scores(0)
        r.close()
        return s
    try:
        if capfd is None:
            return go()
        s, got = traced(capfd, go)
    finally:
        if dense:
            monkeypatch.delenv("RWR_NO_FRONTIER")
    want = 0 if dense else (min(SPARSE_ITERS, n_iter) if sparse is None else sparse)
    assert got == [want], f"seed {seed} n_iter {n_iter}: sparse iterations {got}, expected {want}"
    return s


def top10(a):
    return np.lexsort((np.arange(len(a)), -a))[:10].tolist()


def assert_like_dense(s, d, what):
    assert np.array_equal(s == 0.0, d == 0.0), f"{what}: zero pattern differs from the dense run"
    assert top10(s) == top10(d), f"{what}: top-10 differs from the dense run"
    assert_close_fp64(s, d, what)


@pytest.fixture
def forced(monkeypatch):
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", "1000000")
    monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
    monkeypatch.delenv("RWR_NO_FRONTIER", raising=False)
    return monkeypatch


@pytest.mark.parametrize("case", [(name, N.LAYOUT_AUTO) for name in CASES] +
                         [("uniform6", N.LAYOUT_INDEX), ("uniform6", N.LAYOUT_VALUED)])
def test_one_iteration_is_bit_identical_to_the_oracle(case, forced, capfd):
    name, layout = case
    inp = uniform6() if name == "uniform6" else load_golden(name)["input"]
    gg = gpu_graph(inp, layout=layout)
    assert gg.info().layout == (N.LAYOUT_VALUED if layout == N.LAYOUT_AUTO else layout)
    og = oracle_graph(inp)
    deg = gg.degrees(raw=True)
    for seed in np.flatnonzero(deg > 0)[:6].tolist() + np.flatnonzero(deg == 0)[:2].tolist():
        want, _ = og.run(seed, C015, n_iter=1)
        got = run(gg, seed, 1, capfd=capfd)
        assert np.array_equal(bits(got), bits(want)), f"{name} seed {seed}"
    gg.close()


@pytest.mark.parametrize("name", CASES)
def test_golden_graphs_against_the_oracle_and_the_dense_run(name, forced, capfd):
    g = load_golden(name)
    gg = gpu_graph(g["input"])
    og = oracle_graph(g["input"])
    deg = gg.degrees(raw=True)
    for seed in np.flatnonzero(deg > 0)[:3].tolist():
        for n_iter in (0, 1, 2, 3, 4, 20):
            want, _ = og.run(seed, C015, n_iter=n_iter)
            s = run(gg, seed, n_iter, capfd=capfd)
            assert_close_fp64(s, want, f"{name} seed {seed} n_iter {n_iter}")
            d = run(gg, seed, n_iter, dense=True, monkeypatch=forced, capfd=capfd)
            assert_like_dense(s, d, f"{name} seed {seed} n_iter {n_iter}")
    gg.close()


def test_scale_c2_ninth_against_the_oracle_the_dense_run_and_the_valued_layout(monkeypatch, capfd):
    """A budget of E/64 (the default on graphs above the size floor) forced on a 22 M-link graph: a seed of a few dozen links goes sparse
    for the first iterations; the index-only and the valued layout stay bit-equal."""
    monkeypatch.delenv("RWR_NO_FRONTIER", raising=False)
    monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
    gg = rs.Graph.synthetic(SCALE_C2_NINTH)
    gg.buildGraph()
    assert gg.info().layout == N.LAYOUT_INDEX
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", str(gg.info().nnz // 64))
    gv = rs.Graph.synthetic(SCALE_C2_NINTH, layout=N.LAYOUT_VALUED)
    gv.buildGraph()
    og = oracle_graph(gg.export_links())
    deg = gg.degrees(raw=True)
    seed = int(np.flatnonzero((deg[:SCALE_C2_NINTH["n_users"]] > 10) & (deg[:SCALE_C2_NINTH["n_users"]] < 60))[0])
    n = gg.size()
    for n_iter in (0, 1, 2, 3, 4, 20):
        want, _ = og.run(seed, C015, n_iter=n_iter)
        s = run(gg, seed, n_iter, capfd=capfd)
        assert_close_fp64(s, want, f"n_iter {n_iter}")
        assert abs(s.sum() - n) <= 1e-12 * n
        assert_like_dense(s, run(gg, seed, n_iter, dense=True, monkeypatch=monkeypatch, capfd=capfd), f"n_iter {n_iter}")
        if n_iter == 1:
            assert np.array_equal(bits(s), bits(want))
        if n_iter in (1, 2, 20):
            assert np.array_equal(bits(s), bits(run(gv, seed, n_iter, capfd=capfd))), f"valued layout, n_iter {n_iter}"
    gg.close()
    gv.close()


def test_seed_over_the_budget_stays_dense(monkeypatch, capfd):
    g = load_golden("small_b")
    gg = gpu_graph(g["input"])
    deg = gg.degrees()                          # out-links of the push CSR (raw links after the dedup)
    seed = int(np.argmax(deg))
    monkeypatch.setenv("RWR_FRONTIER_TRACE", "1")
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", str(int(deg[seed])))
    run(gg, seed, 1, capfd=capfd, sparse=1)                             # exactly the budget: sparse
    monkeypatch.setenv("RWR_FRONTIER_BUDGET", str(int(deg[seed]) - 1))
    for n_iter in (1, 2, 5):
        s = run(gg, seed, n_iter, capfd=capfd, sparse=0)
        d = run(gg, seed, n_iter, dense=True, monkeypatch=monkeypatch, capfd=capfd)
        assert np.array_equal(bits(s), bits(d)), f"n_iter {n_iter}"
    gg.close()


def test_dangling_seed_and_seed_with_dangling_neighbours(forced, capfd):
    # seed 0 has only dangling neighbours, 3 is dangling, 5 reaches 4 and 0
    inp = uniform6()
    og = oracle_graph(inp)
    for layout in (N.LAYOUT_INDEX, N.LAYOUT_VALUED):
        gg = gpu_graph(inp, layout=layout)
        assert gg.info().layout == layout
        for seed in (0, 3, 5):
            for n_iter in (0, 1, 2, 3, 4, 9):
                want, _ = og.run(seed, C015, n_iter=n_iter)
                s = run(gg, seed, n_iter, capfd=capfd)
                assert_close_fp64(s, want, f"seed {seed} n_iter {n_iter}")
                d = run(gg, seed, n_iter, dense=True, monkeypatch=forced, capfd=capfd)
                assert_like_dense(s, d, f"seed {seed} n_iter {n_iter}")
        gg.close()


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_large_then_small_neighbourhood_matches_fresh_runs(prec, forced):
    """Reruns on one Model, back to back (the second run of a key captures the iteration graph, every later one replays
    it), seeds with large and small neighbourhoods interleaved; then fresh runs of the same seeds."""
    g = load_golden("small_b")
    gg = gpu_graph(g["input"])
    deg = gg.degrees(raw=True)
    users = np.flatnonzero(deg > 0)
    big, small = int(users[np.argmax(deg[users])]), int(users[np.argmin(deg[users])])
    order = [small, big, small, small, big, big, small]
    for n_iter in (6, 2):
        m = run_fixed(gg, [big], C015, n_iter, prec)
        got = []
        for seed in order:
            m.rerun([seed], C015, n_iter)
            got.append(m.scores(0))
        m.close()
        for seed, s in zip(order, got):
            fresh = run_fixed(gg, [seed], C015, n_iter, prec)
            assert np.array_equal(s, fresh.scores(0)), f"seed {seed} n_iter {n_iter}"
            fresh.close()
    gg.close()


def test_valued_and_index_layouts_bit_equal_at_two_iterations(forced, capfd):
    inp = uniform6()
    gi, gv = gpu_graph(inp, layout=N.LAYOUT_INDEX), gpu_graph(inp, layout=N.LAYOUT_VALUED)
    assert gi.info().layout == N.LAYOUT_INDEX and gv.info().layout == N.LAYOUT_VALUED
    for seed in range(6):
        for prec in (rs.FP64, rs.FP32):
            a, b = run(gi, seed, 2, prec, capfd=capfd), run(gv, seed, 2, prec, capfd=capfd)
            assert np.array_equal(bits(a), bits(b)), f"seed {seed} precision {prec}"
    gi.close()
    gv.close()


@pytest.mark.parametrize("name", CASES)
def test_fp32(name, forced, capfd):
    g = load_golden(name)
    gg = gpu_graph(g["input"])
    og = oracle_graph(g["input"])
    for seed in np.flatnonzero(gg.degrees(raw=True) > 0)[:3].tolist():
        for n_iter in (1, 2, 3, 20):
            want, _ = og.run(seed, C015, n_iter=n_iter)
            f = run(gg, seed, n_iter, rs.FP32, capfd=capfd)
            assert_close_fp32(f, want, f"{name} seed {seed} n_iter {n_iter}")
            d = run(gg, seed, n_iter, rs.FP32, dense=True, monkeypatch=forced, capfd=capfd)
            assert np.array_equal(f == 0.0, d == 0.0)
            assert_close_fp32(f, d, f"{name} seed {seed} n_iter {n_iter} vs dense")
    gg.close()


def test_launch_count_is_the_same_on_the_replayed_graph(forced, capfd):
    g = load_golden("small_a")
    gg = gpu_graph(g["input"])
    seed = int(np.flatnonzero(gg.degrees(raw=True) > 0)[0])
    m, sp = traced(capfd, lambda: run_fixed(gg, [seed], C015, 5))
    assert sp == [SPARSE_ITERS]
    first = m.info().kernel_launches
    assert first > 1 + 3 * 5                     # the frontier kernels are counted
    for _ in range(3):                           # second run captures the graph, later runs replay it
        _, sp = traced(capfd, lambda: m.rerun([seed], C015, 5))
        assert sp == [SPARSE_ITERS]
        assert m.info().kernel_launches == first
    m.close()
    forced.setenv("RWR_NO_FRONTIER", "1")
    d = run_fixed(gg, [seed], C015, 5)
    assert d.info().kernel_launches == 1 + 3 * 5
    d.close()
    gg.close()
