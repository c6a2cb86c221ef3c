#!/usr/bin/env python
"""wavefront_model.py -- CPU MODEL (not a measurement) of what bounds k_spmv_ws: L1TEX wavefronts per gathered link.

The B300/B200 load model (B300_MICROARCH.md, "L1tex wavefront queue") charges a global load instruction one L1TEX cycle
per distinct 128-byte line its 32 lanes touch, and k_spmv_ws is L1TEX-bound (profiles/r01_spmv_ws_fp64_ncu_details.txt).
This script rebuilds, on the CPU with numpy, the label order and the edge stream that graph.cu / stream.cu build for the
bench graph, and counts for every warp-level gather instruction
    * the distinct 128-byte lines among the lanes that go to global memory (labels >= hub entries), and
    * the bank-conflict degree among the lanes that go to the shared-memory hub table (labels < hub entries),
for the stream layout in use and for alternatives that keep the same links but assign them differently to lanes and
instructions.  It needs no GPU and nothing from /root/reference; it uses the CPU oracle's synthetic generator.

    python profiles/microbench/wavefront_model.py [--scale 0.25] [--precision fp64|fp32]

Layouts (a stage is 256 consecutive links of the stream, 8 instructions of 32 lanes):
    lane8             lane L owns links 8L..8L+7 of the stage; instruction k gathers link 8L+k
    lane2             lane L owns links 2L, 2L+1 of a 64-link quarter stage; instruction k gathers 2L+k
    link              instruction i gathers links 32i..32i+31 (lane L <- link 32i+L)
    hybrid  (in use)  link for a stage without a row end (one that lies inside a row), lane8 for every other stage
each with the sources of a row in three orders: original source ascending ("by source", the order before the hybrid
layout), sorted by internal label ("by label"), and sorted by internal label in the rows of more than 256 links only
("long by label", the order in use: shorter rows never fill a stage without a row end).
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

C2_SPEC = dict(seed=20260102, n_users=1_000_000, n_items=10_000_000, n_third=0, authorship_per_mille=1000,
               n_like=76_000_000, n_friend=21_000_000, n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1,
               p1_byte=61, reserved=0)
C4_SPEC = dict(seed=20260104, n_users=5_000_000, n_items=45_000_000, n_third=0, authorship_per_mille=1000,
               n_like=700_000_000, n_friend=200_000_000, n_follow=0, n_mention=0, undefined_per_mille=0, scramble=1,
               p1_byte=61, reserved=0)
HOT_MIN = 8
STAGE = 256


def relabel(n, src, dst):
    """graph.cu:484-528: hot nodes by descending out-degree, cold nodes (1 <= deg < HOT_MIN) clustered by their first
    out-neighbour, nodes without links last."""
    deg = np.bincount(src, minlength=n).astype(np.int64)
    row_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(deg, out=row_ptr[1:])
    order = np.argsort(-deg, kind="stable")                 # old_of_new of the degree sort
    new_of_old = np.empty(n, np.int64)
    new_of_old[order] = np.arange(n)
    n_hot = int((deg >= HOT_MIN).sum())
    cold = np.flatnonzero((deg >= 1) & (deg < HOT_MIN))     # original index order
    if len(cold):
        nb = dst[row_ptr[cold]].astype(np.int64)            # first out-neighbour (original label)
        lab = new_of_old[nb]
        key = np.where(lab < n_hot, lab, n_hot + nb)
        o = np.argsort(key, kind="stable")
        new_of_old[cold[o]] = n_hot + np.arange(len(cold))
    return new_of_old.astype(np.int32), n_hot, deg


def build_stream(n, src, dst, new_of_old, sort_in_row):
    """stream.cu: rows of W^T by ascending internal label, one padding link (label n) for a row without in-links.
    sort_in_row: False (sources in original order), True (by internal label), "long" (by internal label in the rows of
    more than STAGE links only)."""
    row = new_of_old[dst]
    s_lab = new_of_old[src]
    indeg = np.bincount(row, minlength=n)
    if sort_in_row:
        lab = s_lab if sort_in_row is True else np.where(indeg[row] > STAGE, s_lab, 0)
        key = row.astype(np.int64) * (n + 1) + lab
        o = np.argsort(key, kind="stable")
    else:
        o = np.argsort(row, kind="stable")                  # links arrive source-ascending: stable keeps that order
    s_sorted = s_lab[o]
    length = np.maximum(indeg, 1)
    ptr2 = np.zeros(n + 1, np.int64)
    np.cumsum(length, out=ptr2[1:])
    stream = np.full(ptr2[-1], n, np.int32)
    has = indeg > 0
    # positions of real links: row r's links occupy ptr2[r] .. ptr2[r] + indeg[r]
    in_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(indeg, out=in_ptr[1:])
    shift = np.repeat(ptr2[:-1][has] - in_ptr[:-1][has], indeg[has])
    stream[np.arange(len(s_sorted)) + shift] = s_sorted
    return stream


def blocked_stats(n, src, dst, new_of_old, blocks):
    """Column blocking with virtual rows (DESIGN.md section 9): (row, block) pairs that hold links, padding links."""
    row = new_of_old[dst].astype(np.int64)
    blk = new_of_old[src].astype(np.int64) * blocks // n
    pairs = np.unique(row * blocks + blk)
    indeg = np.bincount(row, minlength=n)
    plain = int(np.maximum(indeg, 1).sum())
    virtual = n * blocks
    blocked = len(src) + (virtual - len(pairs))
    return plain, blocked, virtual - len(pairs)


def row_ends(n, dst, new_of_old):
    """[stream links] True on the last link of every row (the end flag of stream.cu)"""
    ptr2 = np.cumsum(np.maximum(np.bincount(new_of_old[dst], minlength=n), 1))
    ends = np.zeros(ptr2[-1], bool)
    ends[ptr2 - 1] = True
    return ends


def instr_matrix(stream, layout, n, ends=None):
    """[instructions, 32] labels, one row per warp-level gather instruction (hybrid: needs the row ends)."""
    pad = (-len(stream)) % STAGE
    s = np.concatenate([stream, np.full(pad, n, np.int32)]) if pad else stream
    if layout == "hybrid":
        st = s.reshape(-1, STAGE)
        e = np.concatenate([ends, np.zeros(pad, bool)]) if pad else ends
        inside = ~e.reshape(-1, STAGE).any(axis=1)        # (the last stage holds the last row end)
        m = np.empty((len(st), STAGE // 32, 32), np.int32)
        m[inside] = st[inside].reshape(-1, STAGE // 32, 32)
        m[~inside] = st[~inside].reshape(-1, 32, 8).transpose(0, 2, 1)
        return m.reshape(-1, 32)
    if layout == "lane8":
        return s.reshape(-1, 32, 8).transpose(0, 2, 1).reshape(-1, 32)
    if layout == "lane2":
        return s.reshape(-1, 32, 2).transpose(0, 2, 1).reshape(-1, 32)
    if layout == "link":
        return s.reshape(-1, 32)
    raise ValueError(layout)


def count(m, hub, elt, chunk=1 << 20):
    """(global wavefronts, shared wavefronts, global lanes, shared lanes) summed over the instructions of m."""
    per_line = 128 // elt
    banks = 32 * 4 // elt                                   # distinct elt-wide bank groups in one shared-memory phase
    g_wf = s_wf = g_l = s_l = 0
    for a in range(0, len(m), chunk):
        x = m[a:a + chunk].astype(np.int64)
        is_s = x < hub
        # global part: distinct lines among the global lanes (shared lanes replaced by a sentinel that is not counted)
        line = np.where(is_s, -1, x // per_line)
        line.sort(axis=1)
        new = np.ones_like(line, dtype=bool)
        new[:, 1:] = line[:, 1:] != line[:, :-1]
        g_wf += int((new & (line >= 0)).sum())
        g_l += int((~is_s).sum())
        # shared part: conflict degree = max over banks of the distinct addresses that hit it
        if hub:
            xs = np.where(is_s, x, -1)
            xs.sort(axis=1)
            first = np.ones_like(xs, dtype=bool)
            first[:, 1:] = xs[:, 1:] != xs[:, :-1]
            first &= xs >= 0
            bank = np.where(first, xs % banks, banks)
            degree = np.zeros(len(xs), np.int64)
            for b in range(banks):
                np.maximum(degree, (bank == b).sum(axis=1), out=degree)
            s_wf += int(degree.sum())
            s_l += int(is_s.sum())
    return g_wf, s_wf, g_l, s_l


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=0.25)
    ap.add_argument("--precision", default="fp64")
    ap.add_argument("--spec", default="c2", choices=["c2", "c4"])
    ap.add_argument("--blocks", type=int, default=0, help="only price column blocking with this many blocks of x")
    args = ap.parse_args()
    import oracle as O

    spec = dict(C2_SPEC if args.spec == "c2" else C4_SPEC)
    for k in ("n_users", "n_items", "n_like", "n_friend"):
        spec[k] = max(4, int(spec[k] * args.scale))
    t0 = time.time()
    g = O.synth_generate(spec)
    n = len(g["node_id"])
    src, dst = g["src"], g["dst"]
    assert (np.diff(src) >= 0).all()
    print(f"graph: n={n} links={len(src)} ({time.time() - t0:.1f} s)", flush=True)
    new_of_old, n_hot, deg = relabel(n, src, dst)
    if args.blocks:
        plain, blocked, pads = blocked_stats(n, src, dst, new_of_old, args.blocks)
        print(f"blocks={args.blocks}: stream {plain} links -> {blocked} links ({pads} padding links of empty (row, block) "
              f"pairs, +{100.0 * (blocked - plain) / plain:.1f} %)")
        return
    elt = 8 if args.precision == "fp64" else 4
    hub_bytes = (99 if elt == 8 else 163) * 1024 - 128
    hub = min((hub_bytes // elt) & ~3, n)
    print(f"n_hot={n_hot}  hub entries={hub}  elt={elt}", flush=True)
    ends = row_ends(n, dst, new_of_old)
    print(f"stages without a row end: {int((~ends[:len(ends) // STAGE * STAGE].reshape(-1, STAGE).any(axis=1)).sum())} "
          f"of {-(-len(ends) // STAGE)}", flush=True)
    print(f"{'order':13s} {'layout':6s} {'links':>11s} {'glob lanes':>11s} {'glob wf':>11s} {'wf/lane':>8s} {'shr lanes':>11s} "
          f"{'shr wf':>10s} {'wf total':>11s} {'wf/link':>8s}")
    for sort_in_row, name in ((False, "by source"), (True, "by label"), ("long", "long by label")):
        stream = build_stream(n, src, dst, new_of_old, sort_in_row)
        for layout in ("lane8", "lane2", "link", "hybrid") if sort_in_row != "long" else ("lane8", "hybrid"):
            m = instr_matrix(stream, layout, n, ends)
            g_wf, s_wf, g_l, s_l = count(m, hub, elt)
            tot = g_wf + s_wf
            print(f"{name:13s} {layout:6s} {len(stream):11d} {g_l:11d} {g_wf:11d} "
                  f"{g_wf / max(g_l, 1):8.3f} {s_l:11d} {s_wf:10d} {tot:11d} {tot / len(stream):8.3f}", flush=True)


if __name__ == "__main__":
    main()
