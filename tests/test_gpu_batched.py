"""The batched request path (K8: k_spmm + k_spmm_fixup + k_spmm_poison in seed tiles of 8 FP64 / 16 FP32 columns) held
node by node, column by column, through rwr_probe_tile_ranks: the rank vectors rwr_recommend (n_seeds >= 2) and
rwr_evaluate_users compute, in original labels.

  every column against the oracle (collapsed form) .... FP64: <= 1e-12 relative per node, the oracle's zeros exactly 0
                                                         FP32: <= 1e-6 normalised L1, the oracle's zeros exactly 0
  a column against the same seed in another tile ...... bit-identical (the bits of column j depend on seed j only)
  NaN / Inf ........................................... per column, the oracle's NaN set and Inf set
  tile top-k (rwr_recommend) ........................... exactly the host selection over the probe's ranks, score bits equal
  evaluation (rwr_evaluate_users) ...................... hits, hits_at_k identical, average precision bit-identical to the
                                                         reference's loop replayed over the probe's ranks
"""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import bits

pytestmark = pytest.mark.gpu

import oracle as O
import recommendersystems_b200 as rs
from recommendersystems_b200 import _native as N
from recommendersystems_b200.rwr import run_fixed

REL = 1e-12
L1_FP32 = 1e-6
C015 = rs.widen_float(0.15)
WIDTH = {rs.FP64: 8, rs.FP32: 16}             # seed columns per SpMM tile (spmm.cu, Vec<T>::B)
CHUNK_ITEMS = 1020                            # path items (rows + links) per merge-path tile (graph.h)
USER, ITEM, ETC = 1, 2, 3
LIKE, FRIENDSHIP, FOLLOW, MENTION = 1, 2, 3, 4


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def probe(g, seeds, n_iter, prec):
    """rwr_probe_tile_ranks -> ranks[len(seeds), N] (original labels, widened to double)"""
    s = np.ascontiguousarray(seeds, np.int32)
    out = np.full((len(s), g.size()), np.nan)
    rc = N.lib().rwr_probe_tile_ranks(g._h, _p(s), len(s), C015, int(n_iter), prec, _p(out))
    assert rc == N.RWR_OK, N.last_error()
    return out


def gpu_graph(inp, **opts):
    g = rs.Graph.from_arrays(inp["node_id"], inp["node_type"], inp["src"], inp["dst"], inp["etype"], inp["w"], **opts)
    g.buildGraph()
    return g


def oracle_graph(inp):
    og = O.OracleGraph(inp["node_id"], inp["node_type"], inp["src"], inp["dst"], inp["etype"], inp["w"])
    assert og.build() == 0
    return og


class Reference:
    """The oracle's rank of (seed, n_iter), computed once"""

    def __init__(self, og):
        self.og, self.memo = og, {}

    def __call__(self, seed, n_iter):
        key = (int(seed), int(n_iter))
        if key not in self.memo:
            self.memo[key] = self.og.run(int(seed), C015, n_iter=int(n_iter))[0]
        return self.memo[key]


def assert_column(got, want, prec, what):
    """The single-seed bars (DESIGN section 4) on one column; NaN and Inf sets must be the oracle's"""
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN set"
    assert np.array_equal(np.isinf(got), np.isinf(want)), f"{what}: Inf set"
    inf = np.isinf(want)
    assert np.array_equal(np.sign(got[inf]), np.sign(want[inf])), f"{what}: sign of Inf"
    fin = np.isfinite(want)
    got, want = got[fin], want[fin]
    zero = want == 0.0
    assert np.all(got[zero] == 0.0), f"{what}: nodes the reference leaves at exactly 0 must stay 0"
    if prec == rs.FP64:
        rel = np.abs(got[~zero] - want[~zero]) / np.abs(want[~zero])
        assert rel.size == 0 or rel.max() <= REL, f"{what}: max rel err {rel.max():.3e}"
    elif want.sum() != 0.0:
        l1 = np.abs(got / got.sum() - want / want.sum()).sum()
        assert l1 <= L1_FP32, f"{what}: normalised L1 {l1:.3e}"


def check_against_oracle(ref, seeds, ranks, n_iter, prec, what=""):
    for j, s in enumerate(seeds):
        assert_column(ranks[j], ref(s, n_iter), prec, f"{what} seed {s} (column {j}) iter {n_iter}")


# ------------------------------------------------------------------------------------------ host selection (Recommender.cs)
def score_key(s):
    """Order-preserving image of a score as System.Double.CompareTo orders it: NaN lowest, -0 == +0"""
    s = np.where(s == 0.0, 0.0, np.asarray(s, np.float64))
    b = s.view(np.uint64)
    k = np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))
    return np.where(np.isnan(s), np.uint64(0), k)


class Candidates:
    """Recommender.cs:14-40 over raw links: ITEM nodes minus the targets of the seed's raw LIKE links"""

    def __init__(self, links):
        self.node_id = np.asarray(links["node_id"], np.int64)
        self.item = np.asarray(links["node_type"]) == ITEM
        src, dst, et = (np.asarray(links[k]) for k in ("src", "dst", "etype"))
        like = et == LIKE
        self.src, self.dst = src[like], dst[like]

    def ranking(self, seed, rank):
        """-> (ids, scores) of the full ranking: score descending (NaN lowest), ties by id descending"""
        cand = self.item.copy()
        cand[self.dst[self.src == seed]] = False
        idx = np.flatnonzero(cand)
        order = np.lexsort((self.node_id[idx], score_key(rank[idx])))[::-1]
        return self.node_id[idx[order]], rank[idx[order]]


def recommend(g, seeds, n_iter, prec, k):
    rec = rs.Recommender(g, precision=prec)
    ids, sc, cnt = rec.RecommendationBatch(seeds, 0.15, n_iter, k)
    return ids, sc, cnt, rec.last_info


def check_topk(g, cands, seeds, n_iter, prec, ks=(1, 2, 10, 16), ranks=None):
    """rwr_recommend returns exactly the host selection over the probe's ranks, with the probe's score bits.
    -> {k: number of columns that overflowed the tile candidate list}"""
    assert len(seeds) >= 2                   # one seed goes through the single-column path
    if ranks is None:
        ranks = probe(g, seeds, n_iter, prec)
    overflow = {}
    for k in ks:
        ids, sc, cnt, info = recommend(g, seeds, n_iter, prec, k)
        for j, s in enumerate(seeds):
            want_ids, want_sc = cands.ranking(s, ranks[j])
            m = min(k, len(want_ids))
            assert cnt[j] == m, (s, k, cnt[j], m)
            assert ids[j, :m].tolist() == want_ids[:m].tolist(), (s, k)
            assert np.array_equal(bits(sc[j, :m]), bits(want_sc[:m])), (s, k)
        B = WIDTH[prec]
        tiles = -(-len(seeds) // B)
        base = tiles * (2 + 3 * n_iter + 5)  # spmm_run_tile + the five top-k launches of a tile (select.cu)
        overflow[k] = (info.kernel_launches - base) // 4
        assert (info.kernel_launches - base) % 4 == 0 and overflow[k] >= 0
    return overflow


# ------------------------------------------------------------------------------------------ merge-path geometry on the host
def merge_path(in_deg):
    """k_partition (iterate.cu) on the host: part[k] = (row, nnz) where the path diagonal k * CHUNK_ITEMS cuts"""
    in_deg = np.asarray(in_deg, np.int64)
    n = len(in_deg)
    in_ptr = np.concatenate([[0], np.cumsum(in_deg)])
    total = n + int(in_ptr[-1])
    n_chunks = max(1, -(-total // CHUNK_ITEMS))
    d = np.minimum(np.arange(n_chunks + 1, dtype=np.int64) * CHUNK_ITEMS, total)
    ends = in_ptr[1:] + np.arange(1, n + 1)            # path position after the end item of row r
    rows = np.searchsorted(ends, d, side="right")       # rows whose end item lies before the diagonal
    return in_ptr, np.stack([rows, d - rows], 1)


def tile_rows(in_ptr, part, k):
    """The rows k_spmm sees in tile k: (row, links in the tile, kind); kind 'whole' (finalised in the tile), 'head' (started
    in an earlier tile, ends here) or 'carry' (continues in the next tile)"""
    n = len(in_ptr) - 1
    (row0, nnz0), (row1, nnz1) = part[k], part[k + 1]
    out = []
    for r in range(row0, min(row1, n - 1) + 1):
        rs_, s = in_ptr[r], max(in_ptr[r], nnz0)
        e = max(in_ptr[r + 1] if r < row1 else nnz1, s)
        kind = "carry" if r >= row1 else ("head" if rs_ < nnz0 else "whole")
        out.append((r, int(e - s), kind))
    return out


def length_class(links):
    return "quad" if links < 32 else ("warp" if links < 256 else "group")


def geometry_input(rng, valued):
    """A graph whose pull CSR (labels = original labels) is laid out to hit every tile case of k_spmm.  -> (input, marks)"""
    deg, marks = [], {}

    def pos():                                           # path position of the next row's first item
        return sum(deg) + len(deg)

    def pad_to(target):                                  # one filler row so that the next row starts at `target` mod CI
        p = (target - pos()) % CHUNK_ITEMS
        if p:
            deg.append(p - 1)

    def row(d, name=None):
        deg.append(d)
        if name:
            marks.setdefault(name, []).append(len(deg) - 1)

    for d in (0, 2, 0, 5):
        row(d)
    for d in (0, 1, 31, 32, 33, 255, 256, 257, 1019, 1020, 1021, 3000, 4000, 5000):
        row(d, f"deg{d}")
        for _ in range(rng.randrange(0, 3)):
            row(rng.randrange(0, 20))
    for d in (5, 31, 32, 100, 256, 600):                 # end item = last item of a tile; the next row starts a tile
        pad_to(CHUNK_ITEMS - 1 - d)
        row(d, "ends_at_tile_end")
        row(40, "starts_at_tile_start")
    for d in (10, 50, 500):                              # last link = last item of a tile: only the row end is left
        pad_to(-d)
        row(d, "only_end_left")
    for d, before in ((40, 20), (300, 100), (700, 300)):  # cut rows whose both parts are in one length class
        pad_to(-before)
        row(d, "cut")
    pad_to(0)
    for _ in range(70):                                  # tiles packed with 32-link rows
        row(32, "packed32")
    pad_to(0)
    for d in (256, 300, 257):                            # three group rows in one tile
        row(d, "three_group")
    while len(deg) < 6_200:                              # enough distinct sources for the 5 000-link row
        row(rng.choice([0, 0, 1, 2, 3, 7]))
    n = len(deg)
    dangling = n - 1                                     # explicit out-degree 0, one raw UNDEFINED link
    marks["dangling"] = [dangling]
    node_type = np.array([(USER, ITEM, ITEM, ETC)[i % 4] for i in range(n)], np.int32)
    node_id = np.asarray(rng.sample(range(100_000, 100_000 + 4 * n), n), np.int64)
    links = []
    pool = np.arange(n - 1)
    nprng = np.random.default_rng(rng.randrange(1 << 30))
    for r, d in enumerate(deg):
        if d == 0:
            continue
        srcs = nprng.choice(pool[pool != r], size=d, replace=False)
        for s in srcs.tolist():
            if node_type[s] == USER and node_type[r] == ITEM:
                t = LIKE
            elif valued and nprng.random() < 0.3:
                t = MENTION
            else:
                t = FRIENDSHIP if nprng.random() < 0.7 else FOLLOW
            w = float(nprng.choice([0.5, 0.25, 1.75, 3 * nprng.random()])) if t == MENTION else 1.0
            links.append((s, r, t, w))
    links.append((dangling, 0, 0, 1.0))
    links.sort(key=lambda x: x[0])                       # grouped by source (stable: insertion order kept)
    src, dst, et, w = (np.array([l[i] for l in links]) for i in range(4))
    inp = dict(node_id=node_id, node_type=node_type, src=src.astype(np.int32), dst=dst.astype(np.int32),
               etype=et.astype(np.int32), w=w.astype(np.float64))
    return inp, marks


def check_geometry(in_deg, marks):
    """Every tile case the graph was laid out for does occur in the merge-path table"""
    in_ptr, part = merge_path(in_deg)
    n_tiles = len(part) - 1
    seen = set()
    long_in_tile, group_in_tile, tiles_of_row = [], [], {}
    for k in range(n_tiles):
        rows = tile_rows(in_ptr, part, k)
        for r, links, kind in rows:
            seen.add((length_class(links), kind))
            tiles_of_row[r] = tiles_of_row.get(r, 0) + 1
        long_in_tile.append(sum(1 for _, l, _ in rows if 32 <= l < 256))
        group_in_tile.append(sum(1 for _, l, _ in rows if l >= 256))
    assert {(c, k) for c in ("quad", "warp", "group") for k in ("whole", "head", "carry")} <= seen, seen
    for d in (0, 1, 31, 32, 33, 255, 256, 257, 1019, 1020, 1021):
        assert (np.asarray(in_deg) == d).any(), d
    assert ((np.asarray(in_deg) >= 3000) & (np.asarray(in_deg) <= 5000)).sum() >= 3
    assert max(tiles_of_row[r] for r in marks["deg5000"]) >= 3                      # a row cut across 3+ tiles
    ends = in_ptr[1:] + np.arange(1, len(in_deg) + 1)
    for r in marks["ends_at_tile_end"]:
        assert ends[r] % CHUNK_ITEMS == 0, r                                         # end item closes a tile
    assert {length_class(in_deg[r]) for r in marks["ends_at_tile_end"]} == {"quad", "warp", "group"}
    starts = {int(part[k][0]) for k in range(1, n_tiles) if part[k][1] == in_ptr[part[k][0]]}
    assert set(marks["starts_at_tile_start"]) <= starts                               # a tile starts at the row's first link
    only_end = {int(part[k][0]) for k in range(1, n_tiles) if part[k][1] == in_ptr[part[k][0] + 1] and in_deg[part[k][0]] > 0}
    assert set(marks["only_end_left"]) <= only_end                                    # links all used up in the tile before
    assert any(part[k][0] == part[k + 1][0] for k in range(n_tiles))                 # a tile inside one row
    assert max(long_in_tile) >= 30                                                    # the fullest long-row list
    assert max(group_in_tile) >= 3                                                    # three rows of >= 256 links
    return in_ptr, part


GEOMETRY = {}


def geometry(variant):
    """variant: 'index' (all weights 1), 'valued' (MENTION weights), 'relabelled' (the valued links, default relabelling)"""
    if variant not in GEOMETRY:
        valued = variant != "index"
        inp, marks = geometry_input(random.Random(4242 if valued else 4141), valued)
        og = oracle_graph(inp)
        opts = dict() if variant == "relabelled" else dict(relabel=False)
        g = gpu_graph(inp, **opts)
        info = g.info()
        assert info.layout == (N.LAYOUT_VALUED if valued else N.LAYOUT_INDEX)
        assert info.relabelled == (variant == "relabelled")
        _, col, _ = og.csr()
        in_deg = np.bincount(col, minlength=og.n)
        in_ptr, part = check_geometry(in_deg, marks)
        assert info.n_chunks == len(part) - 1
        n = og.n
        seeds = []
        for name in ("deg5000", "deg0", "deg1", "deg31", "deg32", "deg33", "deg255", "deg256", "deg257", "deg1019",
                     "deg1020", "deg1021", "deg3000", "deg4000", "ends_at_tile_end", "starts_at_tile_start",
                     "only_end_left", "dangling"):
            seeds += marks[name]
        seeds.insert(3, seeds[0])                        # the same seed twice in one tile
        seeds += [marks["packed32"][35], marks["three_group"][1]]
        rng = random.Random(7)
        while len(seeds) < 40:
            seeds.append(rng.randrange(n))
        raw_out = np.bincount(inp["src"], minlength=n)
        expl_out = np.bincount(inp["src"][inp["etype"] != 0], minlength=n)
        assert in_deg[marks["deg0"][0]] == 0 and raw_out[marks["dangling"][0]] > 0 and expl_out[marks["dangling"][0]] == 0
        GEOMETRY[variant] = dict(inp=inp, g=g, ref=Reference(og), seeds=seeds, marks=marks, cands=Candidates(inp))
    return GEOMETRY[variant]


# ------------------------------------------------------------------------------------------ the probe itself
def test_probe_validates_like_rwr_recommend():
    gm = geometry("index")
    g, n = gm["g"], gm["g"].size()
    L = N.lib()
    out = np.zeros(2 * n)

    def call(seeds, prec=rs.FP64, h=None):
        s = np.asarray(seeds, np.int32)
        return L.rwr_probe_tile_ranks(g._h if h is None else h, _p(s), len(s), C015, 3, prec, _p(out))

    assert L.rwr_probe_tile_ranks(None, None, 0, C015, 3, rs.FP64, None) == N.RWR_E_INVALID
    assert call([0, -1]) == N.RWR_E_INVALID
    assert call([0, n]) == N.RWR_E_BADSEED
    assert call([0, -5]) == N.RWR_E_BADSEED
    assert call([0, 1], prec=7) == N.RWR_E_INVALID
    unbuilt = rs.Graph.from_arrays(gm["inp"]["node_id"], gm["inp"]["node_type"], gm["inp"]["src"], gm["inp"]["dst"],
                                   gm["inp"]["etype"], gm["inp"]["w"])
    assert call([0, 1], h=unbuilt._h) == N.RWR_E_NOT_BUILT
    unbuilt.close()
    # a seed without raw links is a case of the iteration, not an error of it
    f, og, g = nan_graph(NAN_CASES[0])
    no_links = int(np.flatnonzero(np.bincount(f["src"], minlength=og.n) == 0)[0])
    ranks = probe(g, [no_links, 1], 4, rs.FP64)
    assert_column(ranks[0], og.run(no_links, C015, n_iter=4)[0], rs.FP64, "seed without raw links")
    g.close()


# ------------------------------------------------------------------------------------------ (a) every tile case
@pytest.mark.parametrize("variant", ["index", "valued", "relabelled"])
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_tile_cases_every_node_matches_the_oracle(variant, prec):
    gm = geometry(variant)
    seeds = gm["seeds"][:32]
    for n_iter in (1, 2, 7, 20):
        ranks = probe(gm["g"], seeds, n_iter, prec)
        check_against_oracle(gm["ref"], seeds, ranks, n_iter, prec, variant)


# ------------------------------------------------------------------------------------------ (b) tile shapes
@pytest.mark.parametrize("n_iter", [0, 1, 2, 7, 20])
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_tile_shapes(prec, n_iter):
    B = WIDTH[prec]
    for variant in ("index", "valued"):
        gm = geometry(variant)
        for m in (1, B - 1, B, B + 1, 2 * B + 3):
            seeds = gm["seeds"][:m]
            ranks = probe(gm["g"], seeds, n_iter, prec)
            check_against_oracle(gm["ref"], seeds, ranks, n_iter, prec, f"{variant} {m} seeds")


# ------------------------------------------------------------------------------------------ (c) column independence
@pytest.mark.parametrize("variant", ["index", "valued"])
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_a_column_depends_on_its_seed_only(variant, prec):
    gm = geometry(variant)
    g, n = gm["g"], gm["g"].size()
    B = WIDTH[prec]
    seeds = gm["seeds"][:2 * B + 3]
    base = probe(g, seeds, 7, prec)
    assert np.array_equal(bits(probe(g, seeds, 7, prec)), bits(base))               # rerun
    rng = np.random.default_rng(11)
    perm = rng.permutation(len(seeds))                                               # across slots and tiles
    got = probe(g, [seeds[i] for i in perm], 7, prec)
    assert np.array_equal(bits(got), bits(base[perm]))
    for trial in range(2):                                                           # other partners in the tile
        others = rng.integers(0, n, size=3 * len(seeds)).tolist()
        mixed, where = [], []
        for i, s in enumerate(seeds):
            mixed += others[3 * i:3 * i + 1 + trial]
            where.append(len(mixed))
            mixed.append(s)
        got = probe(g, mixed, 7, prec)
        assert np.array_equal(bits(got[where]), bits(base)), trial


# ------------------------------------------------------------------------------------------ (d) NaN / Inf columns
NAN_CASES = [(20260301, 8, 60, 3, 400), (20260302, 12, 90, 4, 700), (20260303, 5, 12, 2, 150)]


def nan_graph(case):
    from random_graphs import random_flat
    seed, *shape = case
    f = random_flat(random.Random(seed), *shape, zero_rows=1, nan_rows=1)
    f = {k: np.asarray(v) for k, v in f.items()}
    og = oracle_graph(f)
    _, _, oval = og.csr()
    assert np.isnan(oval).any() or np.isinf(oval).any()
    return f, og, gpu_graph(f)


@pytest.mark.parametrize("case", NAN_CASES)
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_nan_and_inf_columns_are_the_oracles(case, prec):
    """A row whose weights sum to 0 sends `0 * NaN` to its targets in the first iteration whatever the seed (Model.cs:85-88
    multiplies every rank, zero or not), so every column of such a graph is partly NaN after one iteration and NaN at every
    node after two (k_spmm_poison).  Poisoned columns sit beside the inactive columns of an odd-width last tile, which must
    stay untouched: a wrong bit of the poison mask shows as a column that is not NaN everywhere."""
    f, og, g = nan_graph(case)
    ref = Reference(og)
    n, B = og.n, WIDTH[prec]
    seeds = list(range(n)) + ([0] if n % B % 2 == 0 else [])
    assert len(seeds) % B % 2 == 1
    whole = []
    for n_iter in (1, 2, 3, 8):
        ranks = probe(g, seeds, n_iter, prec)
        check_against_oracle(ref, seeds, ranks, n_iter, prec, f"case {case[0]}")
        whole.append(int(np.isnan(ranks).all(axis=1).sum()))
        # a tile of other partners and another width: the same bits
        sub = seeds[1:B + 2]
        assert np.array_equal(bits(probe(g, sub, n_iter, prec)), bits(ranks[1:B + 2])), n_iter
    assert whole[0] == 0 and whole[1] == len(seeds), whole     # partly NaN after one iteration, NaN everywhere after two
    g.close()


# ------------------------------------------------------------------------------------------ (e) scale
MEDIUM = dict(seed=5, n_users=20_000, n_items=150_000, n_third=5_000, authorship_per_mille=500, n_like=450_000,
              n_friend=120_000, n_follow=20_000, n_mention=3_000, undefined_per_mille=50, scramble=1, p1_byte=40)


def test_medium_graph_hubs_across_hundreds_of_tiles():
    cpu = O.synth_generate(MEDIUM)
    og = oracle_graph(cpu)
    ref = Reference(og)
    g = rs.Graph.synthetic(MEDIUM)
    g.buildGraph()
    info = g.info()
    assert info.max_in_degree > 6_000 and info.n_chunks > 300
    raw_deg = np.bincount(cpu["src"], minlength=og.n)
    _, col, _ = og.csr()
    in_deg = np.bincount(col, minlength=og.n)
    rng = np.random.default_rng(3)
    seeds = [int(np.argmax(raw_deg)), int(np.argmax(in_deg)), int(np.flatnonzero(raw_deg[:MEDIUM["n_users"]] == 1)[0])]
    seeds += rng.choice(np.flatnonzero(raw_deg > 0), size=13, replace=False).tolist()
    for prec in (rs.FP64, rs.FP32):
        s = seeds[:WIDTH[prec]]
        check_against_oracle(ref, s, probe(g, s, 12, prec), 12, prec, "medium")
    g.close()


def test_c2_ninth_one_tile_against_the_oracle():
    """The 1/9-scale C2 graph (22 M links): one FP64 tile of 8 seeds with the largest hub, 20 iterations, every node"""
    spec = dict(seed=11, n_users=120_000, n_items=1_100_000, n_third=0, authorship_per_mille=1000, n_like=7_800_000,
                n_friend=2_200_000, n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1, p1_byte=61)
    g = rs.Graph.synthetic(spec)
    g.buildGraph()
    assert g.info().nnz > 19_000_000
    links = g.export_links()
    og = oracle_graph(links)
    raw_deg = np.bincount(links["src"], minlength=og.n)
    _, col, _ = og.csr()
    rng = np.random.default_rng(5)
    seeds = [int(np.argmax(raw_deg)), int(np.argmax(np.bincount(col, minlength=og.n)))]
    seeds += rng.choice(np.flatnonzero(raw_deg[:spec["n_users"]] > 0), size=6, replace=False).tolist()
    ranks = probe(g, seeds, 20, rs.FP64)
    for j, s in enumerate(seeds):
        want = og.run(s, C015, n_iter=20)[0]
        single = run_fixed(g, [s], C015, 20).scores(0)
        # The seed entry carries the restart mass S, a sum over 1.2 M nodes whose order differs from the reference's
        # sequential one in both device paths: measured 1.07e-12 relative for one of these seeds, in K8 and in the
        # single-seed path alike.  It is held to the single-seed path; every other node to the oracle.
        others = np.arange(og.n) != s
        assert_column(ranks[j][others], want[others], rs.FP64, f"22M-link graph seed {s}")
        assert abs(ranks[j][s] - single[s]) <= REL * abs(single[s]), (s, ranks[j][s], single[s])
        assert abs(ranks[j][s] - want[s]) <= 2 * REL * abs(want[s]), (s, ranks[j][s], want[s])
    g.close()


# ------------------------------------------------------------------------------------------ (f) tile top-k
@pytest.mark.parametrize("variant", ["index", "valued", "relabelled"])
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_tile_topk_is_the_exact_selection_geometry(variant, prec):
    gm = geometry(variant)
    raw_out = np.bincount(gm["inp"]["src"], minlength=gm["g"].size())
    seeds = [s for s in gm["seeds"] if raw_out[s] > 0][:2 * WIDTH[prec] + 3]
    for n_iter in (2, 7):
        check_topk(gm["g"], gm["cands"], seeds, n_iter, prec)


@pytest.mark.parametrize("case", NAN_CASES)
@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_tile_topk_is_the_exact_selection_nan_and_short_lists(case, prec):
    f, og, g = nan_graph(case)
    cands = Candidates(f)
    seeds = np.flatnonzero(np.bincount(f["src"], minlength=og.n) > 0).tolist()
    short = nan_cols = 0
    for n_iter in (1, 3, 8):
        ranks = probe(g, seeds, n_iter, prec)
        check_topk(g, cands, seeds, n_iter, prec, ranks=ranks)
        nan_cols += int(np.isnan(ranks).any(axis=1).sum())
        short += sum(len(cands.ranking(s, ranks[j])[0]) < 16 for j, s in enumerate(seeds))
    assert nan_cols > 0
    if case[2] < 16:
        assert short == 3 * len(seeds)       # every list is shorter than k = 16
    g.close()


def test_tile_topk_overflow_beside_columns_that_fit():
    """After one or two iterations most items tie at exactly 0: a column with fewer than k positive candidates takes more
    than 65 536 candidates at the bound and falls back to the exact per-column path, a column with many does not"""
    spec = dict(seed=31, n_users=2_000, n_items=120_000, n_third=0, authorship_per_mille=300, n_like=60_000, n_friend=4_000,
                n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1, p1_byte=100)
    cpu = O.synth_generate(spec)
    cands = Candidates(cpu)
    g = rs.Graph.synthetic(spec)
    g.buildGraph()
    users = np.flatnonzero(np.bincount(cpu["src"], minlength=len(cpu["node_id"]))[:spec["n_users"]] > 0)[:160].tolist()
    mixed, stats = {rs.FP64: 0, rs.FP32: 0}, []
    for n_iter in (1, 2):
        ranks = probe(g, users, n_iter, rs.FP64)
        positive = np.array([int((cands.ranking(s, ranks[j])[1] > 0).sum()) for j, s in enumerate(users)])
        few = [u for u, p in zip(users, positive) if p < 8]          # fewer than k = 10, 16 blocks hold a positive score
        many = [u for u, p in zip(users, positive) if p >= 40]
        stats.append((n_iter, len(few), len(many), int(positive.max())))
        for prec in (rs.FP64, rs.FP32):
            h = WIDTH[prec] // 2
            if len(few) < h or len(many) < h:
                continue
            seeds = [x for pair in zip(few[:h], many[:h]) for x in pair]             # one tile, interleaved
            over = check_topk(g, cands, seeds, n_iter, prec)
            stats.append((n_iter, prec, over))
            mixed[prec] += sum(0 < over[k] < len(seeds) for k in over)
    assert mixed[rs.FP64] > 0 and mixed[rs.FP32] > 0, stats   # the case under test did occur in both precisions
    g.close()


# ------------------------------------------------------------------------------------------ (g) evaluation
def replay_evaluation(cands, seed, rank, test, k):
    """Experiment.cs:121-128 over the host ranking of the probe's ranks -> (hits, average precision, hits among the first k)"""
    ids, _ = cands.ranking(seed, rank)
    hits, ap = O.evaluate(ids, test)
    return hits, ap, int(np.isin(ids[:k], test).sum())


@pytest.mark.parametrize("prec", [rs.FP64, rs.FP32])
def test_evaluation_is_exact_over_the_tile_ranks(prec):
    import experiment_ref as R
    spec = dict(seed=2024, n_users=4_000, n_items=30_000, n_third=200, authorship_per_mille=900, n_like=260_000,
                n_friend=40_000, n_follow=1_000, n_mention=0, undefined_per_mille=0, scramble=1, p1_byte=61)
    full = O.synth_generate(spec)
    deg_like = np.bincount(full["src"][full["etype"] == LIKE], minlength=len(full["node_id"]))
    users = np.flatnonzero(deg_like[:spec["n_users"]] >= 20)[:45]
    links, test = R.hold_out(full, users, 10, 9)
    g = rs.Graph.from_arrays(full["node_id"], full["node_type"], full["src"], full["dst"], full["etype"], full["w"])
    gtest = g.hold_out(users, 10, 9)
    assert all(gtest[int(u)].tolist() == test[int(u)].tolist() for u in users)
    g.buildGraph()
    cands = Candidates(links)
    n_iter = 15
    ranks = probe(g, users, n_iter, prec)
    if prec == rs.FP64:
        ref = Reference(oracle_graph(links))
        check_against_oracle(ref, users[:4], ranks[:4], n_iter, prec, "hold-out")
    # the held-out sets, and large sets of any node ids (liked items, users, unknown ids) for two tiles of users
    rng = np.random.default_rng(9)
    ids_all = np.asarray(links["node_id"], np.int64)
    big_users = users[:2 * WIDTH[prec]]
    big = {int(u): np.unique(np.concatenate([rng.choice(ids_all, size=3_000 + 500 * (i % 3), replace=False),
                                             ids_all.max() + 1 + np.arange(5)]))
           for i, u in enumerate(big_users)}
    assert sum(len(v) for v in big.values()) > 2048 * 2          # the tiles' items exceed the shared-memory histogram
    total_hits = {}
    for sets, us in ((None, users), (big, big_users)):
        for k in (10, 500):
            r = rs.evaluate_users(g, None if sets is None else us, sets, 0.15, n_iter, k=k, precision=prec)
            for j, u in enumerate(us):
                t = test[int(u)] if sets is None else sets[int(u)]
                hits, ap, atk = replay_evaluation(cands, int(u), ranks[j], t, k)
                assert int(r["hits"][j]) == hits and int(r["hits_at_k"][j]) == atk, (int(u), k)
                assert bits(np.array([r["avg_precision"][j]]))[0] == bits(np.array([ap]))[0], (int(u), k, r["avg_precision"][j], ap)
            total_hits[sets is None, k] = int(r["hits"].sum()), int(r["hits_at_k"].sum())
    assert all(h > 0 and atk > 0 for h, atk in total_hits.values())
    g.close()
