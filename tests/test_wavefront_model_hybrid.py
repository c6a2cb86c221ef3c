"""The hybrid stream layout of the CPU model (profiles/microbench/wavefront_model.py), the one stream.cu builds: a stage
without a row end is stored link-major, every other stage lane-major, and the rows of more than 256 links hold their
sources by label.  On a small graph with long rows: each stage keeps its links, the layouts agree where they must, and the
wavefront counts respect their bounds."""
import importlib.util
import os

import numpy as np

import oracle as O
from conftest import C1_SPEC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("wavefront_model", os.path.join(ROOT, "profiles", "microbench", "wavefront_model.py"))
wm = importlib.util.module_from_spec(spec)
spec.loader.exec_module(wm)


def test_hybrid_layout_and_long_row_order():
    g = O.synth_generate(dict(C1_SPEC, n_mention=0, undefined_per_mille=0, n_like=200_000))
    n, src, dst = len(g["node_id"]), g["src"], g["dst"]
    new_of_old, _, _ = wm.relabel(n, src, dst)
    ends = wm.row_ends(n, dst, new_of_old)
    indeg = np.bincount(new_of_old[dst], minlength=n)
    assert ends.sum() == n and (indeg > 2 * wm.STAGE).any()
    ptr2 = np.concatenate([[0], np.cumsum(np.maximum(indeg, 1))])
    by_source = wm.build_stream(n, src, dst, new_of_old, False)
    long_sorted = wm.build_stream(n, src, dst, new_of_old, "long")
    assert len(ends) == len(by_source) == len(long_sorted)
    for r in range(n):                                      # long rows by label, short rows untouched
        a, b = by_source[ptr2[r]:ptr2[r + 1]], long_sorted[ptr2[r]:ptr2[r + 1]]
        assert np.array_equal(b, np.sort(a) if indeg[r] > wm.STAGE else a)
    per_stage = wm.STAGE // 32
    inside = ~np.concatenate([ends, np.zeros((-len(ends)) % wm.STAGE, bool)]).reshape(-1, wm.STAGE).any(axis=1)
    assert inside.any() and not inside.all()
    for stream in (by_source, long_sorted):
        h = wm.instr_matrix(stream, "hybrid", n, ends).reshape(-1, per_stage, 32)
        l8 = wm.instr_matrix(stream, "lane8", n).reshape(-1, per_stage, 32)
        lk = wm.instr_matrix(stream, "link", n).reshape(-1, per_stage, 32)
        assert np.array_equal(h[inside], lk[inside]) and np.array_equal(h[~inside], l8[~inside])
        assert np.array_equal(np.sort(h.reshape(len(h), -1), axis=1), np.sort(l8.reshape(len(l8), -1), axis=1))
        for hub in (0, 64, 4096):
            g_wf, s_wf, g_l, s_l = wm.count(h.reshape(-1, 32), hub=hub, elt=8)
            assert g_l + s_l == h.size and g_wf <= g_l and s_wf <= s_l and g_wf + s_wf > 0
