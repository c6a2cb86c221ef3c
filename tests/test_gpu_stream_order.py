"""The order of the edge stream inside long rows (stream.cu: k_ws_fill, ws_stage_link): a row of more than 256 links holds
its sources by label, and a 256-link stage without a row end is stored link-major.  The golden graphs have no such
stages; these graphs have a few hub rows of 300 to 5 000 in-links on top of random links, cut by 512-link tiles, so
several flag-free stages sit in every hub row (any 512 consecutive links of a row hold one).  Dense runs
(RWR_NO_FRONTIER=1) go through k_spmv_ws for every iteration."""
import numpy as np
import pytest

from conftest import bits

pytestmark = pytest.mark.gpu

import recommendersystems_b200 as rs
from recommendersystems_b200 import _native as N
from recommendersystems_b200.rwr import run_fixed

from test_gpu_parity import C015, assert_close_fp32, assert_close_fp64, oracle_graph, same_ranking

HUB_IN = (300, 511, 700, 1500, 5000)
N_ITERS = (1, 2, 20)


def hub_graph(seed, n=20_000, n_links=80_000):
    """random links plus hub rows: node h_k gets HUB_IN[k] in-links from distinct sources; one weight per source row
    (all links of one type, weight 1), so that both layouts build"""
    rng = np.random.default_rng(seed)
    src = [rng.integers(0, n, n_links)]
    dst = [rng.integers(0, n, n_links)]
    hubs = rng.choice(n, len(HUB_IN), replace=False)
    for h, d in zip(hubs, HUB_IN):
        src.append(rng.choice(n, d, replace=False))
        dst.append(np.full(d, h))
    src, dst = np.concatenate(src), np.concatenate(dst)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    o = np.argsort(src, kind="stable")
    src, dst = src[o].astype(np.int32), dst[o].astype(np.int32)
    node_type = np.where(np.arange(n) < n // 10, 1, 2).astype(np.int32)
    return dict(node_id=np.arange(n, dtype=np.int64) + 1000, node_type=node_type, src=src, dst=dst,
                etype=np.full(len(src), 2, np.int32), w=np.ones(len(src))), hubs


@pytest.fixture(scope="module", params=[1, 2])
def graphs(request):
    mp = pytest.MonkeyPatch()
    mp.setenv("RWR_TILE_LINKS", "512")
    mp.setenv("RWR_NO_FRONTIER", "1")
    inp, hubs = hub_graph(request.param)
    out = {}
    for layout in (N.LAYOUT_INDEX, N.LAYOUT_VALUED):
        g = rs.Graph.from_arrays(inp["node_id"], inp["node_type"], inp["src"], inp["dst"], inp["etype"], inp["w"], layout=layout)
        g.buildGraph()
        assert g.info().layout == layout
        out[layout] = g
    info = out[N.LAYOUT_INDEX].info()
    assert info.max_in_degree >= max(HUB_IN)
    og = oracle_graph(inp)
    deg = out[N.LAYOUT_INDEX].degrees(raw=True)
    # seeds: two hub sources (their walk reaches a hub row at once), a hub itself when it links out, one node without links
    seeds = [int(s) for s in inp["src"][np.isin(inp["dst"], hubs)][:2]]
    seeds += [int(h) for h in hubs if deg[h] > 0][:1] + [int(np.flatnonzero(deg == 0)[0])]
    yield out, og, seeds
    for g in out.values():
        g.close()
    mp.undo()


def scores(g, seed, n_iter, prec=rs.FP64):
    r = run_fixed(g, [seed], C015, n_iter, prec)
    s = r.scores(0)
    r.close()
    return s


def top10(a):
    return np.lexsort((np.arange(len(a)), -a))[:10]


def test_dense_runs_against_the_oracle(graphs):
    gs, og, seeds = graphs
    for seed in seeds:
        for n_iter in N_ITERS:
            want, _ = og.run(seed, C015, n_iter=n_iter)
            for layout, g in gs.items():
                what = f"seed {seed} n_iter {n_iter} layout {layout}"
                got = scores(g, seed, n_iter)
                assert_close_fp64(got, want, what)
                assert np.array_equal(got == 0.0, want == 0.0), what
                t = top10(got)
                same_ranking(t.tolist(), got[t], top10(want).tolist(), want[top10(want)])
                got32 = scores(g, seed, n_iter, rs.FP32)
                assert np.array_equal(got32 == 0.0, want == 0.0), what + " FP32"
                assert_close_fp32(got32, want, what + " FP32")


def test_layouts_bit_equal_and_reruns_bit_identical(graphs):
    gs, _, seeds = graphs
    gi, gv = gs[N.LAYOUT_INDEX], gs[N.LAYOUT_VALUED]
    for prec in (rs.FP64, rs.FP32):
        for seed in seeds:
            for n_iter in N_ITERS:
                a = scores(gi, seed, n_iter, prec)
                assert np.array_equal(bits(a), bits(scores(gi, seed, n_iter, prec))), (prec, seed, n_iter, "rerun")
                assert np.array_equal(bits(a), bits(scores(gv, seed, n_iter, prec))), (prec, seed, n_iter, "valued layout")
    # Model.rerun on the same result object
    r = run_fixed(gi, [seeds[0]], C015, 20)
    first = r.scores(0)
    r.rerun([seeds[1]], C015, 20)
    r.rerun([seeds[0]], C015, 20)
    assert np.array_equal(bits(r.scores(0)), bits(first))
    r.close()


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_continuation_equals_the_whole_run(graphs, prec):
    gs, _, seeds = graphs
    for g in gs.values():
        for seed in seeds[:2]:
            want = scores(g, seed, 20, prec)
            for a, b in ((1, 19), (7, 13), (19, 1)):
                r = run_fixed(g, [seed], C015, a, prec)
                r.continue_fixed(b)
                assert r.info().iterations == 20
                assert np.array_equal(bits(r.scores(0)), bits(want)), (seed, a, b)
                r.close()
