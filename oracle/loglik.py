"""TEST INFRASTRUCTURE (oracle) -- not product code.

Log-likelihood of given bins under a model, restated from the count tables of oracle.em_read, the priors of
oracle.sampler (bn_dirichlet_prior.m, setTransitionPriors.m) and asub2ind.m, on plain arrays.  It shares nothing with the
packed tables of libemb200 (emb_model.cpp: logp_column) and is what tests/test_loglik.py compares the device code against.

Each conditional is log(w_m / W) with w = N(:, j) + alpha(:, j), the column select_random.m:17 draws from; a zero-total column
gives bin 1 with probability 1 (as the sampler does), a zero-weight bin -inf.
"""
from __future__ import annotations

import numpy as np

from .sampler import bn_dirichlet_prior, set_transition_priors


def logp_table(N, alpha=None) -> np.ndarray:
    """r x q table of log(w_m / W), column by column."""
    w = np.asarray(N, dtype=np.float64) + (0.0 if alpha is None else np.asarray(alpha, dtype=np.float64))
    W = w.sum(axis=0)
    out = np.full(w.shape, -np.inf)
    pos = W > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        lp = np.log(w[:, pos] / W[pos])
    out[:, pos] = np.where(w[:, pos] > 0, lp, -np.inf)
    out[0, ~pos] = 0.0
    return out


def parent_column(G, r, child, X) -> np.ndarray:
    """0-based column j - 1 of asub2ind(r(parents), X(:, parents)) per row of X (1-based bins, one column per variable)."""
    parents = np.nonzero(np.asarray(G, dtype=bool)[:, child])[0]
    if parents.size == 0:
        return np.zeros(X.shape[0], dtype=np.int64)
    siz = np.asarray(r, dtype=np.int64)[parents]
    k = np.concatenate(([1], np.cumprod(siz[:-1])))
    return (np.asarray(X, dtype=np.int64)[:, parents] - 1) @ k


def _alphas(N, prior):
    return bn_dirichlet_prior(N, prior)


def loglik_initial(parms, bins, prior=0):
    """bins: (n, n_initial) 1-based.  Returns (total (n,), per_var (n, n_initial)); per_var summed in variable order."""
    bins = np.asarray(bins, dtype=np.int64)
    alpha = _alphas(parms.N_initial, prior)
    per = np.zeros(bins.shape, dtype=np.float64)
    for i in range(parms.n_initial):
        tab = logp_table(parms.N_initial[i], alpha[i])
        j = parent_column(parms.G_initial, parms.r_initial, i, bins)
        per[:, i] = tab[bins[:, i] - 1, j]
    total = np.zeros(bins.shape[0])
    for i in range(parms.n_initial):
        total = total + per[:, i]
    return total, per


def is_dynvar_depend(parms) -> bool:
    """dbn_sample.m:55: an edge between two (t+1) variables selects the per-step branch."""
    tm = np.asarray(parms.temporal_map)
    G = np.asarray(parms.G_transition, dtype=bool)
    return bool(any(G[a - 1, b - 1] for a in tm[:, 1] for b in tm[:, 1]))


def loglik_tracks(parms, init_bins, bins, prior=0, stay_prior=None, correct_dbn=False):
    """init_bins: (n, n_initial), bins: (n, n_dyn, T), both 1-based (bins[:, d, c] = column c of dynamic variable d, column 0 the
    initial state).  Returns (initial (n,), transition (n,)).  `stay_prior`: setTransitionPriors' value instead of `prior` for
    the transition network."""
    init_bins = np.asarray(init_bins, dtype=np.int64)
    bins = np.asarray(bins, dtype=np.int64)
    n, nd, T = bins.shape
    initial, _ = loglik_initial(parms, init_bins, prior)
    tm = np.asarray(parms.temporal_map)
    r = np.asarray(parms.r_transition)
    if stay_prior is not None:
        alpha = set_transition_priors(parms.G_transition, r, tm, stay_prior)
    else:
        alpha = _alphas(parms.N_transition, prior)
    tabs = [logp_table(parms.N_transition[tm[d, 1] - 1], alpha[tm[d, 1] - 1]) for d in range(nd)]
    frozen = not is_dynvar_depend(parms) and not correct_dbn

    def state(c):
        """full transition-network state for the step into column c (parents at t = column c-1, t+1 = column c)"""
        X = np.ones((n, parms.n_transition), dtype=np.int64)
        X[:, :parms.n_initial] = init_bins
        for d in range(nd):
            X[:, tm[d, 0] - 1] = bins[:, d, c - 1]
            X[:, tm[d, 1] - 1] = bins[:, d, c]
        return X

    transition = np.zeros(n)
    if frozen and T > 1:
        X0 = np.ones((n, parms.n_transition), dtype=np.int64)
        X0[:, :parms.n_initial] = init_bins
        for d in range(nd):
            X0[:, tm[d, 1] - 1] = init_bins[:, tm[d, 0] - 1]
        cols = [parent_column(parms.G_transition, r, tm[d, 1] - 1, X0) for d in range(nd)]
    for c in range(1, T):
        if not frozen:
            X = state(c)
            cols = [parent_column(parms.G_transition, r, tm[d, 1] - 1, X) for d in range(nd)]
        for d in range(nd):
            transition = transition + tabs[d][bins[:, d, c] - 1, cols[d]]
    return initial, transition
