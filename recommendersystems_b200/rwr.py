"""Host-side mirror of `Recommenders.RWRBased` (reference: Recommenders/RWRBased/{Graph,Model,Recommender}.cs).

Same names, argument meaning and error behaviour as the C# classes; every computation is forwarded through the
C ABI of librwr_b200.so (include/rwr_b200.h) -- the same entry points the C# P/Invoke shim binds
(recommendersystems_b200/csharp/RwrNative.cs).  Exceptions map the reference's:
    KeyError    <- KeyNotFoundException   (seed without an `edges` entry, Recommender.cs:21; graph not built, Model.cs:79)
    ValueError  <- ArgumentException      (buildGraph() twice, Graph.cs:86)
    IndexError  <- IndexOutOfRangeException (link target outside the node range, Model.cs:87)
"""
from __future__ import annotations

import ctypes as C
import enum
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N

FP64, FP32 = N.FP64, N.FP32
# initial rank of a restart-set run (include/rwr_b200.h RWR_INIT_*): 1 everywhere, N at one node, fl(N * q_i)
INIT_UNIFORM, INIT_NODE, INIT_RESTART = N.INIT_UNIFORM, N.INIT_NODE, N.INIT_RESTART


class NodeType(enum.IntEnum):      # Recommender.cs:4
    UNDEFINED = 0
    USER = 1
    ITEM = 2
    ETC = 3


class EdgeType(enum.IntEnum):      # Recommender.cs:5
    UNDEFINED = 0
    LIKE = 1
    FRIENDSHIP = 2
    FOLLOW = 3
    MENTION = 4
    AUTHORSHIP = 5
    PURCHASE = 6
    ETC = 7


class RwrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"librwr_b200 error {code}: {msg}")
        self.code = code


def _check(rc: int) -> None:
    if rc == N.RWR_OK:
        return
    msg = N.last_error()
    if rc in (N.RWR_E_BADSEED, N.RWR_E_NOT_BUILT):
        raise KeyError(msg)
    if rc == N.RWR_E_ALREADY_BUILT:
        raise ValueError(msg)
    if rc == N.RWR_E_BADINDEX:
        raise IndexError(msg)
    raise RwrError(rc, msg)


def widen_float(x: float) -> float:
    """`float dampingFactor` widened to double, as Recommender.cs:16 does implicitly (0.15f -> 0.15000000596046448)."""
    return float(np.float32(x))


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Node:                         # Graph.cs:4-17
    __slots__ = ("id", "type")

    def __init__(self, id: int, type: int = NodeType.UNDEFINED):
        self.id = int(id)
        self.type = int(type)


class ForwardLink:                  # Graph.cs:19-35
    __slots__ = ("targetNode", "type", "weight")

    def __init__(self, targetNode: int, type: int = EdgeType.UNDEFINED, weight: float = 1.0):
        self.targetNode = int(targetNode)
        self.type = int(type)
        self.weight = float(weight)

    def __repr__(self):
        return f"ForwardLink({self.targetNode}, {self.type}, {self.weight!r})"


class SynthSpec(dict):
    """Keyword bag for rwr_synth_spec (include/rwr_b200.h)."""
    FIELDS = ("seed", "n_users", "n_items", "n_third", "authorship_per_mille", "n_like", "n_friend", "n_follow",
              "n_mention", "undefined_per_mille", "scramble", "p1_byte", "reserved")

    def to_c(self) -> N.rwr_synth_spec:
        d = dict(n_third=0, authorship_per_mille=1000, n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1,
                 p1_byte=61, reserved=0)
        d.update(self)
        return N.rwr_synth_spec(**{k: int(d[k]) for k in self.FIELDS})


class Methodology(enum.IntEnum):   # TweetRecommender/Experiment.cs:7-15
    BASELINE = 0
    INCL_FRIENDSHIP = 1
    INCL_FOLLOWSHIP_ON_THIRDPARTY = 2
    INCL_AUTHORSHIP = 3
    INCL_MENTIONCOUNT = 4
    INCL_ALLFOLLOWSHIP = 5
    INCL_FRIENDSHIP_AUTHORSHIP = 6
    INCL_FRIENDSHIP_MENTIONCOUNT = 7
    ALL = 8
    EXCL_FRIENDSHIP = 9
    EXCL_FOLLOWSHIP_ON_THIRDPARTY = 10
    EXCL_AUTHORSHIP = 11
    EXCL_MENTIONCOUNT = 12
    INCL_FOLLOWSHIP_ON_THIRDPARTY_AND_AUTHORSHIP = 13
    INCL_FOLLOWSHIP_ON_THIRDPARTY_AND_MENTIONCOUNT = 14
    INCL_AUTHORSHIP_AND_MENTIONCOUNT = 15


class Feature(enum.IntEnum):       # TweetRecommender/Experiment.cs:16
    FRIENDSHIP = 0
    FOLLOWSHIP_ON_THIRDPARTY = 1
    AUTHORSHIP = 2
    MENTIONCOUNT = 3


def methodology_masks(methodology: int) -> Tuple[List[Feature], int, int]:
    """`DataLoader.graphConfiguration(Methodology, fold)` (DataLoader.cs:142-219) + the FRIENDSHIP -> UNDEFINED rewrite of
    Experiment.cs:84-101, as masks over a graph that carries every relation -> (features, undefined_type_mask,
    zero_weight_type_mask); the table itself lives in the native library (rwr_methodology_masks)."""
    f, u, z = C.c_int32(), C.c_int32(), C.c_int32()
    _check(N.lib().rwr_methodology_masks(int(methodology), C.byref(f), C.byref(u), C.byref(z)))
    return [x for x in Feature if f.value >> int(x) & 1], u.value, z.value


def methodology_options(methodology: int) -> dict:
    """Keyword options for `Graph(...)` that turn a full graph into the graph of `methodology`."""
    _, u, z = methodology_masks(methodology)
    return dict(undefined_types=[t for t in EdgeType if u >> int(t) & 1], zero_weight_types=[t for t in EdgeType if z >> int(t) & 1])


def _opts(device=-1, layout=N.LAYOUT_AUTO, relabel=True, hub_entries=-1, batch_width=0, stream=0, kernel=0,
          hot_min_degree=0, undefined_types=(), zero_weight_types=(), x_blocks=0, empty_seed_ok=False) -> N.rwr_opts:
    mask = 0
    for t in undefined_types:            # EdgeType values that count as UNDEFINED at buildGraph() (Experiment.cs:84-101)
        mask |= 1 << int(t)
    zmask = 0
    for t in zero_weight_types:          # EdgeType values whose links keep their slot with weight 0.0 (Methodology 15)
        zmask |= 1 << int(t)
    return N.rwr_opts(device=int(device), layout=int(layout), relabel=0 if relabel else 1, hub_entries=int(hub_entries),
                      batch_width=int(batch_width), kernel=int(kernel), stream=int(stream),
                      hot_min_degree=int(hot_min_degree), undefined_type_mask=mask, zero_weight_type_mask=zmask,
                      x_blocks=int(x_blocks), empty_seed_ok=1 if empty_seed_ok else 0, reserved=0)


class Comm:
    """NCCL communicator of the row-partitioned mode (include/rwr_b200.h `rwr_comm`): one per process / GPU."""

    def __init__(self, rank: int, n_ranks: int, unique_id: bytes, device: int = -1):
        if len(unique_id) != 128:
            raise ValueError("unique_id must be the 128 bytes of Comm.unique_id()")
        self._h = C.c_void_p()
        self.rank, self.n_ranks = int(rank), int(n_ranks)
        o = _opts(device=device)
        buf = C.create_string_buffer(unique_id, 128)
        _check(N.lib().rwr_comm_create(self.rank, self.n_ranks, buf, C.byref(o), C.byref(self._h)))

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(N.lib().rwr_comm_unique_id(buf))
        return buf.raw

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            N.lib().rwr_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Graph:
    """Graph.cs:37-94.  `nodes`: Dictionary<int, Node>; `edges`: Dictionary<int, List<ForwardLink>>."""

    def __init__(self, nodes: Optional[Dict[int, Node]] = None, edges: Optional[Dict[int, List[ForwardLink]]] = None,
                 comm: Optional["Comm"] = None, **opts):
        self._h = C.c_void_p()
        self._opts = opts
        self._comm = comm                 # row-partitioned over the ranks of `comm` (every rank passes the same input)
        self.nodes = nodes
        self.edges = edges
        if nodes is not None:
            # `edges[seed]` throws for a MISSING key only (Recommender.cs:21): an entry with an empty list is served.  The
            # flattened arrays cannot tell the two apart, so the dictionary form checks the key itself (Recommender below)
            self._opts = dict(opts, empty_seed_ok=True)
            n = len(nodes)
            node_id = np.fromiter((nodes[i].id for i in range(n)), np.int64, n)
            node_type = np.fromiter((nodes[i].type for i in range(n)), np.int32, n)
            src, dst, et, w = [], [], [], []
            for i in range(n):                          # `for i in 0..N-1: foreach l in edges[i]`
                for l in (edges or {}).get(i, ()):
                    src.append(i); dst.append(l.targetNode); et.append(l.type); w.append(l.weight)
            self._create(node_id, node_type, np.asarray(src, np.int32), np.asarray(dst, np.int32),
                         np.asarray(et, np.int32), np.asarray(w, np.float64))

    # -- construction -------------------------------------------------------------------------------------------
    def _create(self, node_id, node_type, src, dst, etype, w):
        node_id = np.ascontiguousarray(node_id, np.int64)
        node_type = np.ascontiguousarray(node_type, np.int32)
        src = np.ascontiguousarray(src, np.int32)
        dst = np.ascontiguousarray(dst, np.int32)
        etype = np.ascontiguousarray(etype, np.int32)
        w = np.ascontiguousarray(w, np.float64)
        if not (len(src) == len(dst) == len(etype) == len(w)) or len(node_id) != len(node_type):
            raise ValueError("array lengths differ")
        o = _opts(**self._opts)
        if self._comm is not None:
            _check(N.lib().rwr_graph_create_partitioned(len(node_id), _p(node_id), _p(node_type), len(src), _p(src), _p(dst),
                                                        _p(etype), _p(w), C.byref(o), self._comm._h, C.byref(self._h)))
            return
        _check(N.lib().rwr_graph_create(len(node_id), _p(node_id), _p(node_type), len(src), _p(src), _p(dst), _p(etype),
                                        _p(w), C.byref(o), C.byref(self._h)))

    @classmethod
    def from_arrays(cls, node_id, node_type, src, dst, etype, w, comm: Optional["Comm"] = None, **opts) -> "Graph":
        """Flattened SoA form of (nodes, edges): links grouped by source in insertion order."""
        g = cls(None, None, comm=comm, **opts)
        g._create(node_id, node_type, src, dst, etype, w)
        return g

    @classmethod
    def synthetic(cls, spec: dict, comm: Optional["Comm"] = None, **opts) -> "Graph":
        """Deterministic synthetic graph generated on the device (replaces DataLoader + SQLite)."""
        g = cls(None, None, comm=comm, **opts)
        s = SynthSpec(spec).to_c()
        o = _opts(**opts)
        if comm is not None:
            _check(N.lib().rwr_synth_create_partitioned(C.byref(s), C.byref(o), comm._h, C.byref(g._h)))
        else:
            _check(N.lib().rwr_synth_create(C.byref(s), C.byref(o), C.byref(g._h)))
        return g

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            N.lib().rwr_graph_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference surface --------------------------------------------------------------------------------------
    def buildGraph(self) -> None:
        _check(N.lib().rwr_graph_build(self._h))

    def size(self) -> int:
        return self.info().n_nodes

    # -- probes -------------------------------------------------------------------------------------------------
    def info(self) -> N.rwr_graph_info:
        i = N.rwr_graph_info()
        _check(N.lib().rwr_graph_get_info(self._h, C.byref(i)))
        return i

    def csr(self) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """`Graph.graph` as (row_ptr[N+1], targetNode[nnz], weight[nnz]); null rows are empty."""
        i = self.info()
        if not i.built:
            raise KeyError("buildGraph() has not run")
        rp = np.empty(i.n_nodes + 1, np.int64)
        col = np.empty(i.nnz, np.int32)
        val = np.empty(i.nnz, np.float64)
        _check(N.lib().rwr_graph_get_csr(self._h, _p(rp), _p(col), _p(val)))
        return rp, col, val

    def csr_types(self) -> np.ndarray:
        """`graph[i][k].type` of every explicit link, CSR order (Graph.cs:73-74 keeps the whole ForwardLink)."""
        i = self.info()
        if not i.built:
            raise KeyError("buildGraph() has not run")
        t = np.empty(i.nnz, np.int32)
        _check(N.lib().rwr_graph_get_csr_types(self._h, _p(t)))
        return t

    def hold_out(self, users: Sequence[int], n_folds: int, fold: int) -> Dict[int, np.ndarray]:
        """`DataLoader.splitLikeHistory` (DataLoader.cs:122-140) on the device for every user of `users`: the LIKE links
        (both directions) of the fold's tweets leave `edges`; -> {user: held-out tweet ids, ascending} (`loader.testSet`).
        Call before buildGraph()."""
        u = np.ascontiguousarray(users, np.int32)
        if len(u) and (u.min() < 0 or u.max() >= self.size()):
            raise KeyError("user outside the node range")
        cap = int(self.degrees(raw=True)[u].sum()) if len(u) else 0     # a user's test set is a subset of its raw links
        ptr = np.zeros(len(u) + 1, np.int64)
        ids = np.empty(max(cap, 1), np.int64)
        total = C.c_int64()
        _check(N.lib().rwr_graph_hold_out(self._h, _p(u), len(u), int(n_folds), int(fold), _p(ptr), _p(ids), cap, C.byref(total)))
        self.test_users, self.test_ptr, self.test_ids = u, ptr, ids[:total.value].copy()
        return {int(x): self.test_ids[ptr[i]:ptr[i + 1]] for i, x in enumerate(u)}

    def degrees(self, raw: bool = False) -> np.ndarray:
        n = self.info().n_nodes
        d = np.empty(n, np.int32)
        if raw:
            _check(N.lib().rwr_graph_get_degrees(self._h, None, _p(d)))
        else:
            _check(N.lib().rwr_graph_get_degrees(self._h, _p(d), None))
        return d

    def export_links(self) -> dict:
        i = self.info()
        out = dict(node_id=np.empty(i.n_nodes, np.int64), node_type=np.empty(i.n_nodes, np.int32),
                   src=np.empty(i.n_links_raw, np.int32), dst=np.empty(i.n_links_raw, np.int32),
                   etype=np.empty(i.n_links_raw, np.int32), w=np.empty(i.n_links_raw, np.float64))
        _check(N.lib().rwr_graph_export_links(self._h, _p(out["node_id"]), _p(out["node_type"]), _p(out["src"]),
                                              _p(out["dst"]), _p(out["etype"]), _p(out["w"])))
        return out


class _Result:
    def __init__(self, h: C.c_void_p, n_seeds: int, n_nodes: int, graph: "Graph"):
        self._h, self.n_seeds, self.n_nodes = h, n_seeds, n_nodes
        self._graph = graph               # keeps the native graph alive for as long as its results exist

    def close(self):
        if self._h is not None and self._h.value:
            N.lib().rwr_result_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> N.rwr_run_info:
        i = N.rwr_run_info()
        _check(N.lib().rwr_result_get_info(self._h, C.byref(i)))
        return i

    def rerun(self, seeds: Sequence[int], c: float, n_iter: int) -> None:
        """The same Model object run again from its constructor state with other seeds; no device allocation."""
        s = np.ascontiguousarray(seeds, np.int32)
        if len(s) != self.n_seeds:
            raise ValueError("rerun() needs the same number of seeds")
        _check(N.lib().rwr_rerun_fixed(self._h, _p(s), float(c), int(n_iter)))

    def continue_fixed(self, n_iter: int) -> None:
        """`Model.run(int)` again: n_iter more iterations of every slot from the rank it holds, bit-identical to one run of
        the total count (n_iter <= 0: nothing)."""
        _check(N.lib().rwr_continue_fixed(self._h, int(n_iter)))

    def continue_threshold(self, thr: float = 0.0, max_iter: int = 0) -> np.ndarray:
        """`Model.run(double)` (thr <= 0: `Model.run()`) from the rank every slot holds -> iterations of this call per slot."""
        it = np.zeros(self.n_seeds, np.int32)
        _check(N.lib().rwr_continue_threshold(self._h, float(thr), int(max_iter), _p(it)))
        return it

    def set_rank(self, slot: int, v) -> None:
        """`model.rank = v`: the next continuation of `slot` starts from v (N doubles, original labels)."""
        a = np.ascontiguousarray(v, np.float64)
        if a.shape != (self.n_nodes,):
            raise ValueError(f"rank must hold {self.n_nodes} values")
        _check(N.lib().rwr_set_rank(self._h, int(slot), _p(a)))

    def scores(self, slot: int = 0) -> np.ndarray:
        out = np.empty(self.n_nodes, np.float64)
        _check(N.lib().rwr_scores(self._h, slot, _p(out)))
        return out

    def topk(self, k: int):
        ids = np.zeros((self.n_seeds, k), np.int64)
        sc = np.zeros((self.n_seeds, k), np.float64)
        cnt = np.zeros(self.n_seeds, np.int32)
        _check(N.lib().rwr_topk(self._h, k, _p(ids), _p(sc), _p(cnt)))
        return ids, sc, cnt

    def rank_all(self, slot: int = 0, cap: Optional[int] = None):
        cap = self.n_nodes if cap is None else cap
        ids = np.empty(cap, np.int64)
        sc = np.empty(cap, np.float64)
        cnt = C.c_int64()
        _check(N.lib().rwr_rank_all(self._h, slot, _p(ids), _p(sc), cap, C.byref(cnt)))
        m = min(cnt.value, cap)
        return ids[:m], sc[:m], cnt.value


def run_fixed(graph: Graph, seeds: Sequence[int], c: float, n_iter: int, precision: int = FP64) -> _Result:
    s = np.ascontiguousarray(seeds, np.int32)
    h = C.c_void_p()
    _check(N.lib().rwr_run_fixed(graph._h, _p(s), len(s), float(c), int(n_iter), precision, C.byref(h)))
    return _Result(h, len(s), graph.size(), graph)


def run_threshold(graph: Graph, seeds: Sequence[int], c: float, thr: float, max_iter: int = 0, precision: int = FP64):
    s = np.ascontiguousarray(seeds, np.int32)
    it = np.zeros(len(s), np.int32)
    h = C.c_void_p()
    _check(N.lib().rwr_run_threshold(graph._h, _p(s), len(s), float(c), float(thr), int(max_iter), precision, _p(it),
                                     C.byref(h)))
    return _Result(h, len(s), graph.size(), graph), it


def _restart_args(nodes: Sequence[int], weights: Sequence[float]):
    n = np.ascontiguousarray(nodes, np.int32)
    w = np.ascontiguousarray(weights, np.float64)
    if n.ndim != 1 or n.shape != w.shape:
        raise ValueError("one weight per node")
    return n, w


def run_fixed_restart(graph: Graph, nodes: Sequence[int], weights: Sequence[float], c: float, n_iter: int,
                      init: int = INIT_RESTART, init_node: int = 0, precision: int = FP64) -> _Result:
    """`Model.restart` = `weights` at `nodes` (0 elsewhere, not normalised), then run(n_iter): a walk that restarts over a
    weighted node set (personalized PageRank with a preference vector).  `init`: the initial rank, INIT_UNIFORM (1
    everywhere), INIT_NODE (N at `init_node`) or INIT_RESTART (fl(N * weight)).  One rank vector (slot 0); its top-k and
    ranking exclude the LIKE targets of every listed node."""
    n, w = _restart_args(nodes, weights)
    h = C.c_void_p()
    _check(N.lib().rwr_run_fixed_restart(graph._h, _p(n), _p(w), len(n), int(init), int(init_node), float(c), int(n_iter),
                                         precision, C.byref(h)))
    return _Result(h, 1, graph.size(), graph)


def run_threshold_restart(graph: Graph, nodes: Sequence[int], weights: Sequence[float], c: float, thr: float,
                          max_iter: int = 0, init: int = INIT_RESTART, init_node: int = 0, precision: int = FP64):
    """run_fixed_restart with Model.run(double threshold) (Model.cs:57-66) -> (result, iterations)."""
    n, w = _restart_args(nodes, weights)
    it = np.zeros(1, np.int32)
    h = C.c_void_p()
    _check(N.lib().rwr_run_threshold_restart(graph._h, _p(n), _p(w), len(n), int(init), int(init_node), float(c), float(thr),
                                             int(max_iter), precision, _p(it), C.byref(h)))
    return _Result(h, 1, graph.size(), graph), int(it[0])


class Model:
    """Model.cs:5-116.  `Model(graph, d)` = uniform restart, `Model(graph, d, targetNode)` = seeded.  `restart` (Model.cs:9)
    may be assigned an N-vector: every run then restarts over its nonzeros.  The Model keeps its live result on the device:
    `run(int)` and `run(double)` continue from the rank it holds (`run(5); run(5)` is `run(10)`, bit for bit), and an
    assigned `rank` (Model.cs:7) is where the next run starts -- a warm start.  On a row-partitioned graph, or after
    `restart` changed since the last run, a run starts from the constructor state instead: run(int) for the run(int) and
    updateRanks() iterations so far (threshold iterations are not replayed), and run(double) raises NotImplementedError once
    either has run.  A rank cannot be written on a row-partitioned graph."""

    def __init__(self, graph: Graph, dampingFactor: float, targetNode: Optional[int] = None, precision: int = FP64):
        self.graph = graph
        self.nNodes = graph.size()
        self.dampingFactor = float(dampingFactor)
        self.targetNode = targetNode
        self.precision = precision
        self.nIterations = 0              # deliverRanks() calls so far
        self._fixed_total = 0             # run(int) and updateRanks() iterations so far: the count a fallback run replays
        self._res: Optional[_Result] = None
        self._res_restart: Optional[np.ndarray] = None   # `restart` as it was when _res ran
        self._delivered: Optional[np.ndarray] = None     # deliverRanks() has advanced _res: the rank before it
        self._held: Optional[np.ndarray] = None          # a host copy of the rank _res holds (None: not read since it changed)
        self.residual = float("nan")
        self.nextRank = np.zeros(self.nNodes)         # Model.cs:8
        self._restart: Optional[np.ndarray] = None    # None: the constructor's restart vector

    def _seed(self) -> int:
        return -1 if self.targetNode is None else int(self.targetNode)

    def _set(self):
        """the nonzeros of an assigned `restart` that differs from the constructor's, else None"""
        if self._restart is None or np.array_equal(self._restart, self._constructor_restart()):
            return None
        nz = np.flatnonzero(self._restart)
        return nz, self._restart[nz]

    def _run_fixed(self, n_iter: int) -> _Result:
        s = self._set()
        if s is None:
            return run_fixed(self.graph, [self._seed()], self.dampingFactor, n_iter, self.precision)
        init = INIT_UNIFORM if self.targetNode is None else INIT_NODE
        return run_fixed_restart(self.graph, s[0], s[1], self.dampingFactor, n_iter, init, max(self._seed(), 0), self.precision)

    def _fresh(self, n_iter: int) -> None:
        """the live result becomes a run of n_iter iterations from the constructor state"""
        self._res = self._run_fixed(n_iter)
        self._held = None
        self._res_restart = None if self._restart is None else self._restart.copy()

    def _live(self) -> bool:
        """the live result can be continued: it exists, the graph is not row-partitioned, `restart` has not changed"""
        if self._res is None or self.graph._comm is not None:
            return False
        a, b = self._res_restart, self._restart
        return (a is None and b is None) or (a is not None and b is not None and np.array_equal(a, b))

    def _settle(self) -> None:
        """a deliverRanks() without its updateRanks(): `rank` is still the rank before it, put it back"""
        if self._delivered is not None:
            prev, self._delivered = self._delivered, None
            self._res.set_rank(0, prev)
            self._held = prev
            self.nextRank = np.zeros(self.nNodes)

    def run(self, arg=None, max_iter: int = 0) -> None:
        """run(int nIterations) / run(double threshold) / run() -- Model.cs:68-73, :57-66, :52-55."""
        self._settle()
        self._held = None
        if isinstance(arg, (int, np.integer)) and not isinstance(arg, bool):
            n = max(int(arg), 0)
            self._fixed_total += n
            if self._live():
                self._res.continue_fixed(n)
                self.nIterations += n
            else:
                self._fresh(self._fixed_total)
                self.nIterations = self._fixed_total
            return
        thr = 0.0 if arg is None else float(arg)      # thr <= 0 selects Model.run(): (1/double.MaxValue) * N
        if self._live():
            self.nIterations += int(self._res.continue_threshold(thr, max_iter)[0])
        else:
            if self._fixed_total:
                raise NotImplementedError("threshold run after run(int) / updateRanks() on a row-partitioned graph or after "
                                          "`restart` changed")
            s = self._set()
            self._res_restart = None if self._restart is None else self._restart.copy()
            if s is None:
                self._res, it = run_threshold(self.graph, [self._seed()], self.dampingFactor, thr, max_iter, self.precision)
                self.nIterations = int(it[0])
            else:
                init = INIT_UNIFORM if self.targetNode is None else INIT_NODE
                self._res, self.nIterations = run_threshold_restart(self.graph, s[0], s[1], self.dampingFactor, thr, max_iter,
                                                                    init, max(self._seed(), 0), self.precision)
        self.residual = self._res.info().residual

    # -- the step methods of Model.cs:76-115: each deliverRanks() / updateRanks() pair is one iteration on the device
    def _constructor_restart(self) -> np.ndarray:     # Model.cs:25, :45-48
        r = np.zeros(self.nNodes)
        if self.targetNode is None:
            r[:] = 1.0 / self.nNodes
        else:
            r[self.targetNode] = 1.0
        return r

    @property
    def restart(self) -> np.ndarray:      # Model.cs:9
        return self._constructor_restart() if self._restart is None else self._restart

    @restart.setter
    def restart(self, value) -> None:
        r = np.array(value, np.float64)
        if r.shape != (self.nNodes,):
            raise ValueError(f"restart must hold {self.nNodes} weights")
        self._settle()
        self._restart = r

    def deliverRanks(self) -> None:
        """nextRank = one iteration from rank; rank is unchanged.  A second call before updateRanks() changes nothing."""
        if self._delivered is not None:
            return
        if self._res is None:
            self._fresh(0)
        if not self._live():                          # from the constructor state, O(step) per call
            res = self._run_fixed(self._fixed_total + 1)
            self.nextRank = res.scores(0)
            res.close()
            return
        self._delivered = self._held if self._held is not None else self._res.scores(0)
        self._res.continue_fixed(1)
        self.nextRank = self._held = self._res.scores(0)

    def updateRanks(self) -> None:
        """rank = nextRank: the iteration deliverRanks() computed (without it, one iteration is computed here)."""
        self._fixed_total += 1
        if self._delivered is not None:
            self._delivered = None
            self.nIterations += 1
        elif self._live():
            self._held = None
            self._res.continue_fixed(1)
            self.nIterations += 1
        else:
            self._fresh(self._fixed_total)
            self.nIterations = self._fixed_total
        self.nextRank = np.zeros(self.nNodes)

    def checkConvergence(self, threshold: float) -> bool:
        diff = 0.0
        for a, b in zip(self.rank.tolist(), self.nextRank.tolist()):     # sequential, like Model.cs:111-113
            diff += abs(a - b)
        return diff < threshold

    @property
    def rank(self) -> np.ndarray:
        if self._delivered is not None:
            return self._delivered
        if self._res is None:             # constructor state, Model.cs:24 / :44
            r = np.ones(self.nNodes) if self.targetNode is None else np.zeros(self.nNodes)
            if self.targetNode is not None and 0 <= self.targetNode < self.nNodes:
                r[self.targetNode] = self.nNodes
            return r
        return self._res.scores(0)

    @rank.setter
    def rank(self, value) -> None:
        """`model.rank = v` (Model.cs:7): the next run starts from v (a warm start).  Not on a row-partitioned graph."""
        v = np.array(value, np.float64)
        if v.shape != (self.nNodes,):
            raise ValueError(f"rank must hold {self.nNodes} values")
        if self.graph._comm is not None:
            raise RwrError(N.RWR_E_UNSUPPORTED, "a rank cannot be written on a row-partitioned graph")
        self._delivered = None
        self.nextRank = np.zeros(self.nNodes)
        if not self._live():
            self._fresh(0)
        self._res.set_rank(0, v)
        self._held = None


class Recommender:
    """Recommender.cs:7-52."""

    def __init__(self, graph: Graph, precision: int = FP64):
        self.graph = graph
        self.precision = precision
        self.last_info = None

    def Recommendation(self, idxTargetUser: int, dampingFactor: float, nIteration: int,
                       topN: Optional[int] = None) -> List[Tuple[int, float]]:
        """`dampingFactor` is the reference's C# float: it is widened to double here, as at Recommender.cs:16."""
        c = widen_float(dampingFactor)
        if self.graph.edges is not None and int(idxTargetUser) not in self.graph.edges:
            raise KeyError(f"edges has no entry for node {idxTargetUser} (KeyNotFoundException, Recommender.cs:21)")
        if topN is not None and 0 < topN <= 16:
            # fused request path: seed in, top-k (id, score) pairs out, nothing else crosses the boundary
            ids, sc, cnt = self.RecommendationBatch([int(idxTargetUser)], dampingFactor, nIteration, int(topN))
            m = int(cnt[0])
            return list(zip(ids[0, :m].tolist(), sc[0, :m].tolist()))
        res = run_fixed(self.graph, [int(idxTargetUser)], c, int(nIteration), self.precision)
        try:
            self.last_info = res.info()
            if topN is not None and topN > 0:
                ids, sc, cnt = res.topk(int(topN))
                m = int(cnt[0])
                return list(zip(ids[0, :m].tolist(), sc[0, :m].tolist()))
            # 3-argument overload; the 4-argument one returns the whole list too when topN <= 0 (Recommender.cs:47)
            ids, sc, _ = res.rank_all(0)
            return list(zip(ids.tolist(), sc.tolist()))
        finally:
            res.close()

    def RecommendationForSet(self, nodes: Sequence[int], weights: Sequence[float], dampingFactor: float, nIteration: int,
                             topN: Optional[int] = None) -> List[Tuple[int, float]]:
        """Not in the reference: the ranking for a weighted node set -- a group of users, a session of items -- from a Model
        whose `restart` is `weights` at `nodes`, initial rank fl(N * weight).  The candidates are the ITEM nodes none of the
        listed nodes has liked (Recommender.cs:20-24 for each of them), in the (score desc, id desc) order of
        Recommender.cs:34-38; topN > 0 keeps the first topN.  `dampingFactor` is widened from float as in Recommendation."""
        res = run_fixed_restart(self.graph, nodes, weights, widen_float(dampingFactor), int(nIteration), INIT_RESTART, 0,
                                self.precision)
        try:
            self.last_info = res.info()
            if topN is not None and topN > 0:
                ids, sc, cnt = res.topk(int(topN))
                m = int(cnt[0])
                return list(zip(ids[0, :m].tolist(), sc[0, :m].tolist()))
            ids, sc, _ = res.rank_all(0)
            return list(zip(ids.tolist(), sc.tolist()))
        finally:
            res.close()

    def RecommendationBatch(self, seeds: Iterable[int], dampingFactor: float, nIteration: int, topN: int):
        """n x Recommendation(seed, c, nIter, topN) through the fused tiled path -> (ids[n,k], scores[n,k], counts[n])."""
        s = np.ascontiguousarray(list(seeds), np.int32)
        ids = np.zeros((len(s), topN), np.int64)
        sc = np.zeros((len(s), topN), np.float64)
        cnt = np.zeros(len(s), np.int32)
        info = N.rwr_run_info()
        _check(N.lib().rwr_recommend(self.graph._h, _p(s), len(s), widen_float(dampingFactor), int(nIteration),
                                     self.precision, int(topN), _p(ids), _p(sc), _p(cnt), C.byref(info)))
        self.last_info = info
        return ids, sc, cnt


def evaluate_users(graph: Graph, users: Optional[Sequence[int]] = None, test: Optional[Dict[int, Sequence[int]]] = None,
                   dampingFactor: float = 0.15, nIteration: int = 20, k: int = 10, precision: int = FP64):
    """Experiment.cs:121-128 for many users on the device (rwr_evaluate_users): for every user the number of hits and the
    average precision over the FULL ranking `Recommendation(user, dampingFactor, nIteration)`, plus the hits among the first
    k.  `users` / `test` None: the users and test sets of `graph.hold_out(...)`.
    -> dict(hits, avg_precision, hits_at_k, n_test: arrays [n_users]; info)"""
    if users is None:
        u, ptr, ids = graph.test_users, graph.test_ptr, graph.test_ids
    else:
        u = np.ascontiguousarray(users, np.int32)
        if test is None:
            t = dict(zip(graph.test_users.tolist(), range(len(graph.test_users))))
            sets = [graph.test_ids[graph.test_ptr[t[int(x)]]:graph.test_ptr[t[int(x)] + 1]] for x in u]
        else:
            sets = [np.asarray(list(test[int(x)]), np.int64) for x in u]
        ptr = np.zeros(len(u) + 1, np.int64)
        np.cumsum([len(x) for x in sets], out=ptr[1:])
        ids = np.ascontiguousarray(np.concatenate(sets) if sets else np.zeros(0), np.int64)
    ptr = np.ascontiguousarray(ptr, np.int64)
    ids = np.ascontiguousarray(ids, np.int64)
    n = len(u)
    hits = np.zeros(n, np.int32); atk = np.zeros(n, np.int32); nt = np.zeros(n, np.int32); ap = np.zeros(n, np.float64)
    info = N.rwr_run_info()
    _check(N.lib().rwr_evaluate_users(graph._h, _p(u), n, _p(ptr), _p(ids) if len(ids) else None, widen_float(dampingFactor),
                                      int(nIteration), precision, int(k), _p(hits), _p(ap), _p(atk), _p(nt), C.byref(info)))
    return dict(hits=hits, avg_precision=ap, hits_at_k=atk, n_test=nt, info=info)


def evaluate(recommendation: Sequence[Tuple[int, float]], testSet: Iterable[int]) -> Tuple[int, float]:
    """Experiment.cs:121-128, :136 -> (nHits, averagePrecision)."""
    ids = np.ascontiguousarray([p[0] for p in recommendation], np.int64)
    t = np.ascontiguousarray(list(testSet), np.int64)
    hits, ap = C.c_int32(), C.c_double()
    _check(N.lib().rwr_evaluate(_p(ids), len(ids), _p(t), len(t), C.byref(hits), C.byref(ap)))
    return hits.value, ap.value
