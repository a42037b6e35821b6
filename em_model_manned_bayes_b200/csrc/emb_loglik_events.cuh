// emb_loglik_events.cuh -- log-likelihood of tracks given as event lists (the rows of emb_sample_track_events[_packed]): the
// per-track routine of k_loglik_events (emb_kernels.cu).  __host__ __device__ like emb_loglik.cuh, so that tests/emu runs it too.
//
// The result is defined by reduction: scoring a list equals emb_loglik_tracks on the dense bins the list expands to
// (events2samples.m:9-27: a row is visible from column sum(dt up to and including it) on, of several rows setting one variable in
// one column the last wins, closing rows and rows at column >= T change nothing, a list with sum(dt) < T holds its last state).
// Bins only change at rows, so the walk costs O(rows) instead of O(T): the track is cut into runs of columns over which the
// dynamic state is constant, and each run is scored at once.
//  - frozen branch: run lengths go into the same per-(variable, bin) counters as loglik_transition_frozen, and the same
//    (d, b)-ordered sum (loglik_frozen_sum) turns them into the term -- the counts are exact integers, so the result is
//    bit-identical to the dense scoring.
//  - per-step branch: the first column of a run is the step from the previous state, every further column scores the same
//    slots, so a run adds lp(prev -> run) once and dmul(length - 1, lp(run -> run)), in time order.  This differs from the
//    dense second-by-second sum only in rounding (the tests bound it at 1e-12 relative).
#pragma once
#include "emb_loglik.cuh"

namespace emb {

// status bits of the event-list scoring, beside LL_BAD_BIN / LL_BAD_COL0 (emb_api.cpp: loglik_status_error)
constexpr int32_t LL_BAD_VAR = 4;       // a variable id outside 0..n_initial (8-byte rows) or a gated ordinal above n_gated (packed)
constexpr int32_t LL_BAD_STATIC = 8;    // a row of a static variable with a bin other than its init_bins value
constexpr int32_t LL_BAD_OFFSETS = 16;  // offsets negative or decreasing

struct EventRows {
    const int64_t* offsets;   // [n+1]: the rows of track s are [offsets[s], offsets[s+1])
    const uint32_t* words;    // 8-byte rows: emb_event as word pairs, the first dt | var << 16 | bin << 24; packed rows: the words
    const uint8_t* dts;       // packed rows: dt & 255
};

EMB_HD uint32_t ll_ldg32(const uint32_t* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// row k -> dt, 0-based variable (-1: closing row, -2: no such variable) and 1-based bin (emb200.h: emb_event and the packed word)
template <bool PACKED>
EMB_HD void ll_event_row(const DevModel& M, const EventRows& R, int64_t k, uint32_t& dt, int& v, uint32_t& bin) {
    if (PACKED) {
        const uint32_t w = ll_ldg32(R.words + k);
#if defined(__CUDA_ARCH__)
        dt = (uint32_t)__ldg(R.dts + k) | ((w >> 30) << 8);
#else
        dt = (uint32_t)R.dts[k] | ((w >> 30) << 8);
#endif
        const int g = (int)((w >> 27) & 7u);
        v = g == 0 ? -1 : g > M.n_gated ? -2 : M.gated_var[g - 1];
        bin = ((w >> 23) & 15u) + 1u;
    } else {
        const uint32_t w = ll_ldg32(R.words + 2 * k);
        dt = w & 0xFFFFu;
        const int var = (int)((w >> 16) & 0xFFu);
        v = var == 0 ? -1 : var > M.n_initial ? -2 : var - 1;
        bin = w >> 24;
    }
}

// dynamic ordinal of initial variable v (0-based), -1 for a static variable
EMB_HD int ll_dyn_of(const DevModel& M, int v) {
    for (int d = 0; d < M.n_dyn; ++d)
        if (M.dyn_t[d] == v) return d;
    return -1;
}

EMB_HD uint32_t ll_byte(uint64_t state, int d) { return (uint32_t)(state >> (8 * d)) & 0xFFu; }

// Whole track s: initial term (loglik_initial_one), column-0 check, transition term on the branch `frozen` selects.
// dyn_of[v] = ll_dyn_of(M, v) for every initial variable; cnt as in loglik_transition_frozen.
template <bool PACKED, class Cnt>
EMB_HD void loglik_track_events(const DevModel& M, const LoglikParams& P, const EventRows& R, const int8_t* dyn_of, int64_t s,
                                bool frozen, Cnt cnt) {
    uint8_t x[MAXX];
    for (int i = 0; i < MAXX; ++i) x[i] = 0;
    const double init = loglik_initial_one(M, M.logp_init, P, s, x);
    if (P.initial) P.initial[s] = init;
    const int nd = M.n_dyn, T = P.T;
    int cbase[MAXD];
    int k = 0;
    for (int d = 0; d < nd; ++d) {
        cbase[d] = k;
        if (frozen)
            for (int b = 0; b < M.dyn[d].r; ++b) cnt(k + b) = 0;
        k += M.dyn[d].r;
    }
    // dynamic state: byte d = 0-based bin of dynamic variable d
    uint64_t s0 = 0;
    for (int d = 0; d < nd; ++d) s0 |= (uint64_t)x[M.dyn_t[d]] << (8 * d);
    uint64_t cur = s0;    // state after the rows read so far
    uint64_t run = s0;    // state of the current run, which starts at column rs
    uint64_t prev = s0;   // state of column rs - 1
    int t = 0, rs = 0;    // column the rows read so far are visible at (saturated at T)
    int32_t bad = 0;
    double acc = 0.0;

    // adds the run [rs, re) of state `run`, entered from `prev`
    auto close = [&](int re) {
        if (frozen) {
            const int len = re - (rs > 1 ? rs : 1);
            if (len > 0)
                for (int d = 0; d < nd; ++d) cnt(cbase[d] + (int)ll_byte(run, d)) += (uint32_t)len;
            return;
        }
        if (rs >= 1) {   // column rs: parents at time t see the previous state
            for (int d = 0; d < nd; ++d) {
                x[M.dyn_t[d]] = (uint8_t)ll_byte(prev, d);
                x[M.dyn_t1[d]] = (uint8_t)ll_byte(run, d);
            }
            for (int d = 0; d < nd; ++d) acc = dadd(acc, ldg64(M.logp_trans + ll_column(M.dyn[d], x) + x[M.dyn_t1[d]]));
        }
        const int len = re - rs - 1;   // columns rs+1 .. re-1 (1 .. re-1 for the run that starts at column 0)
        if (len > 0) {
            for (int d = 0; d < nd; ++d) x[M.dyn_t[d]] = x[M.dyn_t1[d]] = (uint8_t)ll_byte(run, d);
            for (int d = 0; d < nd; ++d)
                acc = dadd(acc, dmul((double)len, ldg64(M.logp_trans + ll_column(M.dyn[d], x) + x[M.dyn_t1[d]])));
        }
    };
    // the rows read so far complete column t (< T): its state is cur
    auto column_done = [&]() {
        if (t == 0) {
            if (cur != s0) bad |= LL_BAD_COL0;
        } else if (cur != run) {
            close(t);
            prev = run;
            run = cur;
            rs = t;
        }
    };

    int64_t a = R.offsets[s], e = R.offsets[s + 1];
    if (a < 0 || e < a || e > R.offsets[P.n]) {
        bad |= LL_BAD_OFFSETS;
        e = a;
    }
    for (int64_t q = a; q < e; ++q) {
        uint32_t dt, bin;
        int v;
        ll_event_row<PACKED>(M, R, q, dt, v, bin);
        if (dt && t < T) {
            column_done();
            t = (int)dt < T - t ? t + (int)dt : T;
        }
        if (v == -1) continue;
        if (v == -2) {
            bad |= LL_BAD_VAR;
            continue;
        }
        const int d = dyn_of[v];
        if (d >= 0) {
            uint32_t b0 = bin - 1u;
            if (b0 >= (uint32_t)M.dyn[d].r) {
                bad |= LL_BAD_BIN;
                b0 = 0;
            }
            if (t < T) cur = (cur & ~(0xFFull << (8 * d))) | ((uint64_t)b0 << (8 * d));
        } else if (bin - 1u >= (uint32_t)M.init[v].r) {
            bad |= LL_BAD_BIN;
        } else if (bin != (uint32_t)x[v] + 1u) {
            bad |= LL_BAD_STATIC;
        }
    }
    if (t < T) column_done();
    close(T);
    if (bad) ll_flag(P.status, bad);
    if (!P.transition) return;
    if (frozen) {
        for (int d = 0; d < nd; ++d) x[M.dyn_t1[d]] = x[M.dyn_t[d]] = (uint8_t)ll_byte(s0, d);
        acc = loglik_frozen_sum(M, x, cnt);
    }
    P.transition[s] = acc;
}

}  // namespace emb
