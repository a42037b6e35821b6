"""Seeded synthetic models at the compiled limits of include/emb200.h (EMB_MAX_VARS 24, EMB_MAX_DYN 8, EMB_MAX_PARENTS 8,
EMB_MAX_GATED 16, 127 bins), written in the reference's file grammar through em_write.  The shipped models stay far inside
those limits, so these are what reach the device branches only such models take: k_tracks_generic with 5-8 dynamic variables
and a permuted gate order, 8-byte event rows with 4-bit gated ordinals, the shrunken block of the frozen-branch scoring
kernels, k_initial_fast fp32 entries read from global memory, 128-slot columns, histograms at 64 bins, the shared-memory
staging threshold of the initial kernels, and a fast kernel shape on a model it was not written for.

Every model is a pure function of its seed.  Count columns all have a positive sum; some bins have zero weight and some
columns a single nonzero bin.  Boundaries mix edges straddling zero (a zero bin), '*' variables, edges spanning many orders
of magnitude, and single bins straddling zero (no zero bin: the value can cancel, so the fp32 entries are refused)."""
from __future__ import annotations

import os

import numpy as np

from em_model_manned_bayes_b200.em_write import em_write


def _counts(rs, r, q):
    """r x q count table with zero-weight bins and single-bin columns; every column sums to > 0"""
    N = rs.randint(1, 60, size=(r, q)).astype(np.float64)
    N[rs.random_sample((r, q)) < 0.3] = 0.0
    for j in range(q):
        if r > 1 and (rs.random_sample() < 0.15 or N[:, j].sum() == 0):
            N[:, j] = 0.0
            N[rs.randint(r), j] = rs.randint(1, 30)
    N[0, N.sum(axis=0) == 0] = 1.0
    return N


def _edges(rs, kind, r):
    """r + 1 bin edges of one kind ('*' gives none)"""
    if kind == "*":
        return []
    if kind == "zero":                                      # one bin straddles zero: em_read's zero bin
        e = np.concatenate(([0.0], np.cumsum(rs.uniform(0.25, 4.0, r))))
        k = rs.randint(r) if r > 1 else 0
        return list(np.round(e - (e[k] + e[k + 1]) / 2.0 + rs.uniform(-0.1, 0.1) * (e[k + 1] - e[k]), 6))
    if kind == "wide":                                      # positive edges spanning ~18 orders of magnitude
        return list(np.geomspace(1e-6, 1e12, r + 1) * rs.uniform(0.5, 2.0))
    if kind == "span":                                      # one bin straddling zero without a zero bin (needs > 2 edges)
        assert r == 1
        return [-rs.uniform(1e3, 1e9), rs.uniform(1e3, 1e12)]
    raise ValueError(kind)


def _write(path, seed, r, edges, kinds, rates, dyn=(), trans=None):
    """r: bins per initial variable; edges: (parent, child) of the initial network (0-based); kinds: boundary kind per
    variable; rates: resample rates; dyn: 0-based dynamic variables (ascending); trans: {k: parents of the (t+1) node of
    dynamic variable k}, parents as transition-network indices (i < n: variable i at t; n + j: dynamic variable j at t+1)."""
    rs = np.random.RandomState(seed)
    n = len(r)
    G = np.zeros((n, n), dtype=int)
    for p, c in edges:
        G[p, c] = 1

    def q_of(Gm, rr, c):
        return int(np.prod([rr[p] for p in np.nonzero(Gm[:, c])[0]])) if Gm[:, c].any() else 1

    N_i = [_counts(rs, r[i], q_of(G, r, i)) for i in range(n)]
    kw = dict(labels_initial=['"x%d"' % (i + 1) for i in range(n)], G_initial=G, r_initial=r, N_initial=N_i,
              boundaries=[_edges(rs, kinds[i], r[i]) for i in range(n)], resample_rates=rates)
    if dyn:
        nd = len(dyn)
        rt = list(r) + [r[v] for v in dyn]
        Gt = np.zeros((n + nd, n + nd), dtype=int)
        for k in range(nd):
            for p in trans[k]:
                Gt[p, n + k] = 1
        kw.update(labels_transition=['"x%d(t)"' % (i + 1) if i in dyn else '"x%d"' % (i + 1) for i in range(n)] +
                  ['"x%d(t+1)"' % (v + 1) for v in dyn],
                  G_transition=Gt, r_transition=rt, N_transition=[None] * n + [_counts(rs, rt[n + k], q_of(Gt, rt, n + k))
                                                                               for k in range(nd)])
    return em_write(path, **kw)


def wide_frozen(path):
    """24 initial variables, 8 dynamic ones of 100-127 bins with no dynamic -> dynamic edge (frozen branch), 16 gated, a
    non-identity topological order, a fp64-only single-bin variable"""
    n = 24
    dyn = [2, 5, 8, 11, 14, 17, 20, 23]
    r = [3, 4, 127, 2, 40, 120, 3, 5, 113, 2, 4, 108, 6, 2, 104, 3, 1, 101, 2, 4, 100, 3, 2, 116]
    kinds = ["zero", "*", "zero", "wide", "zero", "*", "zero", "wide", "wide", "*", "zero", "zero",
             "wide", "*", "*", "zero", "span", "wide", "zero", "*", "zero", "wide", "zero", "*"]
    rates = [0.0] * n
    for k, v in enumerate([0, 3, 6, 9, 12, 15, 18, 21]):   # 8 resampled variables, interleaved with the dynamic ones
        rates[v] = [0.01, 0.2, 0.05, 0.5, 0.003, 0.1, 0.9, 0.04][k]
    for k, v in enumerate(dyn):
        rates[v] = 0.0 if k % 3 else 0.07
    edges = [(4, 1), (6, 3), (9, 7), (13, 12), (21, 19), (1, 10), (15, 0), (19, 22), (3, 4), (18, 16)]
    trans = {k: [v] + ([[0, 3, 9, 13][k // 2]] if k % 2 else []) for k, v in enumerate(dyn)}
    return _write(path, 101, r, edges, kinds, rates, dyn, trans)


def deep_step(path):
    """20 initial variables, 8 dynamic ones with dynamic parents (per-step branch) in a topological order that is not the
    file order, (t+1) nodes with 8 parents, 12 gated variables of <= 16 bins with resampled variables after dynamic ones"""
    n = 20
    dyn = [1, 4, 6, 9, 11, 13, 15, 17]
    r = [2, 4, 16, 2, 3, 2, 5, 2, 3, 7, 2, 3, 40, 4, 9, 6, 2, 8, 11, 13]
    kinds = ["zero", "*", "zero", "wide", "zero", "*", "zero", "wide", "zero", "wide", "*", "zero",
             "wide", "zero", "*", "zero", "zero", "wide", "*", "zero"]
    rates = [0.0] * n
    for v, a in ((0, 0.3), (2, 0.05), (18, 0.7), (19, 0.02)):
        rates[v] = a
    for k, v in enumerate(dyn):
        rates[v] = [0.1, 0.0, 0.02, 0.0, 0.5, 0.0, 0.0, 0.2][k]
    edges = [(0, 3), (3, 5), (5, 8), (2, 7), (7, 10), (12, 16), (14, 19), (16, 18)]
    D = {k: n + k for k in range(8)}                       # (t+1) node of dynamic variable k
    trans = {0: [1, D[7], 0, 3, 5, 7, 8, 10],              # 8 parents, one of them a (t+1) node
             1: [4, D[3], 16],
             2: [6, D[5]],
             3: [9, 2],
             4: [11, D[1], 0, 5, 7, 8, 10, 16],            # 8 parents
             5: [13],
             6: [15, D[2], 3],
             7: [17, D[6]]}
    return _write(path, 202, r, edges, kinds, rates, dyn, trans)


def init15_wide(path):
    """15 initial variables in identity order, 280 bins in all, one variable of 127 bins (128-slot columns); no
    transition network"""
    r = [5, 30, 12, 3, 20, 127, 8, 2, 16, 9, 4, 25, 6, 3, 10]
    kinds = ["zero", "wide", "*", "zero", "wide", "zero", "*", "zero", "wide", "zero", "*", "zero", "wide", "*", "zero"]
    edges = [(0, 5), (0, 2), (2, 4), (3, 6), (5, 7), (7, 9), (1, 10), (6, 12), (8, 13), (11, 14), (5, 14), (9, 11)]
    return _write(path, 303, r, edges, kinds, [0.0] * 15)


def hist64(path, bins=64):
    """a 64-bin dynamic variable and a 64-bin static one: the histogram stride exactly (bins=65: one past it)"""
    r = [bins, 3, bins, 5]
    trans = {0: [0, 1], 1: [3]}
    return _write(path, 404 + bins, r, [(1, 0), (3, 2)], ["zero", "*", "wide", "zero"], [0.0, 0.0, 0.2, 0.05], [0, 3], trans)


# Two 15-variable initial networks of 4-slot columns (every r <= 4): the staged table (8 words per column with the pad)
# and the fp64 log-probability table (8 bytes per slot) are both 8 * 4 bytes per column, so 3072 columns are exactly
# 96 KB (staged) and 3073 one column over (gathered from global memory) for k_initial_fast and k_loglik_initial alike.
STAGING = {
    "staging_under": ([2, 1, 4, 3, 4, 3, 4, 4, 4, 3, 2, 3, 4, 4, 2],
                      [[], [], [], [0, 1], [0, 1], [2, 3], [5], [2, 4], [1, 5], [1], [2, 3, 5, 8, 9], [1, 9], [9],
                       [1, 3, 4, 5, 6, 7, 12], [5, 8, 10, 11, 12]]),
    "staging_over": ([4, 1, 2, 4, 4, 4, 1, 4, 3, 4, 3, 2, 4, 4, 2],
                     [[], [0], [0, 1], [1], [2], [], [2, 4], [3], [0, 2, 6], [0, 5, 6], [3, 4, 5, 6], [2, 4, 5, 7, 9, 10],
                      [0, 2, 3, 7], [3, 6, 8, 9, 10], [0, 2, 6, 7, 8, 9, 10]]),
}


def staging(path, name):
    r, parents = STAGING[name]
    kinds = ["*" if ri == 1 else ["zero", "wide", "*"][i % 3] for i, ri in enumerate(r)]
    return _write(path, 505 + len(name), r, [(p, c) for c, ps in enumerate(parents) for p in ps], kinds, [0.0] * 15)


def fast_shape_twin(path, step=False):
    """dynamic variables of 5, 7, 7 bins and no other gated variable: the shape (0x070705, NG 3) of the 7-variable uncor
    models, on a model with other parents, boundaries, rates and variable positions.  step: a (t+1) -> (t+1) edge making the
    sampling order (1, 2, 0), the per-step shape of glider_v1 and its relatives"""
    r = [3, 5, 4, 7, 2, 7]
    kinds = ["*", "zero", "wide", "zero", "zero", "wide"]
    trans = {0: [1, 2] + ([6 + 2] if step else []), 1: [3, 0], 2: [5, 4]}
    return _write(path, 606 + step, r, [(0, 2), (4, 5), (2, 3)], kinds, [0.0, 0.15, 0.0, 0.6, 0.0, 0.03], [1, 3, 5], trans)


# name -> (writer, what the case must reach).  The tests assert each of these from the loaded model.
CASES = {
    "wide_frozen": (wide_frozen, "k_tracks_generic (8 dynamic), frozen scoring with a block < 128 and > 96 KB of shared "
                                 "memory, histograms refused (r > 64), event rows refused (bins > 16)"),
    "deep_step": (deep_step, "k_tracks_generic with a permuted gate_of_dyn and order_dyn; 8-byte event rows with 4-bit "
                             "gated ordinals; packed rows refused; per-step scoring; 8 control and 8 transition.txt columns"),
    "init15_wide": (init15_wide, "k_initial_fast<15> with fp32 entries read from global memory (> 256 bins); 128-slot "
                                 "columns"),
    "hist64": (hist64, "histograms at exactly HIST_STRIDE = 64 bins"),
    "staging_under": (lambda p: staging(p, "staging_under"), "k_initial_fast / k_loglik_initial staged table at 96 KB"),
    "staging_over": (lambda p: staging(p, "staging_over"), "k_initial_fast / k_loglik_initial gather, 96 KB + 32 bytes"),
    "fast_shape_twin": (fast_shape_twin, "specialised kernel (0x070705, 3, frozen) on a model it was not written for"),
    "fast_shape_twin_step": (lambda p: fast_shape_twin(p, step=True),
                             "specialised kernel (0x070705, 3, per-step, order 1 2 0) on a model it was not written for"),
}


def write_all(directory):
    """Write every case (and the 65-bin twin of hist64) into `directory`; returns {name: path}."""
    os.makedirs(directory, exist_ok=True)
    out = {}
    for name, (writer, _) in CASES.items():
        out[name] = writer(os.path.join(directory, name + ".txt"))
    out["hist65"] = hist64(os.path.join(directory, "hist65.txt"), bins=65)
    return out
