"""TEST INFRASTRUCTURE (oracle) -- not product code.

Log-likelihood of tracks given as event lists, restated independently of libemb200: every list is expanded on its own, row by
row, the way events2samples.m:9-27 replays it, and the dense bins are scored second by second by oracle.loglik.loglik_tracks.
tests/test_loglik_events.py compares the event-list scoring of emb_loglik_events.cuh against it.
"""
from __future__ import annotations

import numpy as np

from .loglik import loglik_tracks


def expand_track_events(init_row, dt, var, bins, T):
    """events2samples.m:9-27 for one track, row by row: (n_initial,) initial bins and the rows' dt, var (1-based, 0 = closing
    row) and bin -> n_initial x T bins.  Each row lets the state hold dt more seconds, then sets its variable from that column
    to the end (a later row overwrites); rows at column >= T are dropped."""
    X = np.repeat(np.asarray(init_row, dtype=np.int64)[:, None], T, axis=1)
    t = 0
    for d, v, b in zip(dt, var, bins):
        t += int(d)
        if int(v) > 0 and t < T:
            X[int(v) - 1, t:] = int(b)
    return X


def loglik_track_events(parms, init_bins, dt, var, bins, offsets, T, prior=0, stay_prior=None, correct_dbn=False):
    """init_bins: (n, n_initial); dt / var / bins: the rows of all tracks back to back, track s owning rows
    offsets[s]:offsets[s+1].  Every track is expanded on its own (expand_track_events) and scored second by second
    (loglik_tracks).  Returns (initial (n,), transition (n,))."""
    init_bins = np.asarray(init_bins, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    n = init_bins.shape[0]
    tm = np.asarray(parms.temporal_map)
    dense = np.zeros((n, tm.shape[0], T), dtype=np.int64)
    for s in range(n):
        a, b = offsets[s], offsets[s + 1]
        X = expand_track_events(init_bins[s], dt[a:b], var[a:b], bins[a:b], T)
        dense[s] = X[tm[:, 0] - 1]
    return loglik_tracks(parms, init_bins, dense, prior=prior, stay_prior=stay_prior, correct_dbn=correct_dbn)
