// emb_loglik.cuh -- log-likelihood of given bins under a model: the per-sample scoring routines of k_loglik_initial and
// k_loglik_tracks (emb_kernels.cu).  __host__ __device__ like emb_device.cuh, so that tests/emu runs the same code on the CPU.
//
// The tables are HostModel::logp_initial / logp_transition: log(w_m / W) in fp64, computed on the host by the packer
// (emb_model.cpp: logp_column) at exactly the slots of the threshold tables, so Node::off, rp and stride_rp address them.
// The device only gathers, counts, multiplies and adds (round-to-nearest, no contraction), so device and host agree bit for bit.
#pragma once
#include <cstring>

#include "emb_device.cuh"

namespace emb {

// status bits of the scoring kernels (emb_api.cpp: loglik_status_error)
constexpr int32_t LL_BAD_BIN = 1;    // a bin outside 1..r
constexpr int32_t LL_BAD_COL0 = 2;   // tile column 0 differs from init_bins of the dynamic variables

struct LoglikParams {
    int64_t n;
    int32_t T;
    const int8_t* init_bins;   // [n_initial][n], 1-based
    const int8_t* bins;        // tracks: [ceil(T/4)][ceil(n/128)][n_dyn][128][4], 1-based (emb200.h: emb_track_out)
    double* initial;           // [n] initial term (nullable for tracks)
    double* per_var;           // [n_initial][n] per-variable initial terms (nullable; initial network only)
    double* transition;        // [n] transition term (nullable)
    int32_t* status;           // LL_* bits
};

EMB_HD void ll_flag(int32_t* status, int32_t bit) {
#if defined(__CUDA_ARCH__)
    atomicOr(status, bit);
#else
    *status |= bit;
#endif
}

// offset of the column of `nd` selected by the parents in x (asub2ind.m:13-14 times rp), in table slots
EMB_HD uint32_t ll_column(const Node& nd, const uint8_t* x) {
    uint32_t o = nd.off;
    for (int p = 0; p < nd.np; ++p) o += nd.stride_rp[p] * (uint32_t)x[nd.par[p]];
    return o;
}

// bins of four consecutive seconds of one variable (byte j = second 4*grp + j) as one 32-bit load; offsets are multiples of 4
EMB_HD uint32_t ll_load4(const int8_t* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(reinterpret_cast<const unsigned int*>(p));
#else
    uint32_t v;
    std::memcpy(&v, p, 4);
    return v;
#endif
}

// Reads the initial bins of sample s into x (0-based) and returns sum_i log p(x_i | parents), summed in variable order.
// `logp`: the initial table (global or shared memory).  A bin outside 1..r raises LL_BAD_BIN and is scored as bin 1.
EMB_HD double loglik_initial_one(const DevModel& M, const double* logp, const LoglikParams& P, int64_t s, uint8_t* x) {
    const int n = M.n_initial;
    for (int i = 0; i < n; ++i) {
        int b = P.init_bins[(int64_t)i * P.n + s];
        if (b < 1 || b > M.init[i].r) {
            ll_flag(P.status, LL_BAD_BIN);
            b = 1;
        }
        x[i] = (uint8_t)(b - 1);
    }
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
        const double lp = logp[ll_column(M.init[i], x) + x[i]];
        if (P.per_var) P.per_var[(int64_t)i * P.n + s] = lp;
        acc = dadd(acc, lp);
    }
    return acc;
}

// Column 0 of the tiles of track s against the initial bins in x (0-based).
EMB_HD void loglik_check_col0(const DevModel& M, const LoglikParams& P, int64_t s, const uint8_t* x) {
    const int64_t ntile = num_tiles(P.n);
    for (int d = 0; d < M.n_dyn; ++d) {
        const int b = P.bins[tile_offset(M.n_dyn, ntile, d, 0, s)];
        if (b != (int)x[M.dyn_t[d]] + 1) ll_flag(P.status, LL_BAD_COL0);
    }
}

// The frozen-branch transition term from the counters: sum over (variable d, bin b) of count(d, b) * logp[col_d + b], in (d, b)
// order, counter k = (sum of r over the variables before d) + b.  x: the initial bins, dynamic (t+1) slots set to their time-t bins.
template <class Cnt>
EMB_HD double loglik_frozen_sum(const DevModel& M, const uint8_t* x, Cnt cnt) {
    double acc = 0.0;
    int k = 0;
    for (int d = 0; d < M.n_dyn; ++d) {
        const uint32_t col = ll_column(M.dyn[d], x);
        for (int b = 0; b < M.dyn[d].r; ++b) {
            const uint32_t c = cnt(k + b);
            if (c) acc = dadd(acc, dmul((double)c, ldg64(M.logp_trans + col + b)));   // c == 0 skipped: 0 * -inf is NaN
        }
        k += M.dyn[d].r;
    }
    return acc;
}

// Frozen-parent branch (dbn_sample.m:110-135): the column of every dynamic variable is fixed by column 0, so the transition term is
// sum over (variable d, bin b) of count(d, b) * logp[col_d + b], the counts taken over columns 1..T-1 and the sum in (d, b) order.
// cnt(k) is the counter k = cbase[d] + b of this track (thread-private; shared memory [k][thread] on the device).
// x: the initial bins of the track (0-based), dynamic (t+1) slots set to their time-t bins.
template <class Cnt>
EMB_HD double loglik_transition_frozen(const DevModel& M, const LoglikParams& P, int64_t s, const uint8_t* x, Cnt cnt) {
    const int nd = M.n_dyn, T = P.T;
    const int64_t ntile = num_tiles(P.n);
    int cbase[MAXD];
    int k = 0;
    for (int d = 0; d < nd; ++d) {
        cbase[d] = k;
        for (int b = 0; b < M.dyn[d].r; ++b) cnt(k + b) = 0;
        k += M.dyn[d].r;
    }
    bool bad = false;
    const int ngrp = (T + 3) >> 2;
    for (int grp = 0; grp < ngrp; ++grp) {
        const int c0 = grp * 4;
        for (int d = 0; d < nd; ++d) {
            const uint32_t w = ll_load4(P.bins + tile_offset(nd, ntile, d, grp, s));
            const uint32_t r = (uint32_t)M.dyn[d].r;
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + j;
                if (c == 0 || c >= T) continue;
                const uint32_t b = ((w >> (8 * j)) & 0xFFu) - 1u;   // int8 bins 1..r; anything else wraps above r - 1
                if (b < r) cnt(cbase[d] + (int)b) += 1u;
                else bad = true;
            }
        }
    }
    if (bad) ll_flag(P.status, LL_BAD_BIN);
    return loglik_frozen_sum(M, x, cnt);
}

// Per-step branch (dbn_sample.m:66-79, or correct_dbn): at column c the parents see the time-t slots at column c-1 and the (t+1)
// slots at column c; sum over c = 1..T-1, then d, in that order.  x: the initial bins of the track (0-based), modified.
EMB_HD double loglik_transition_step(const DevModel& M, const LoglikParams& P, int64_t s, uint8_t* x) {
    const int nd = M.n_dyn, T = P.T;
    const int64_t ntile = num_tiles(P.n);
    uint32_t last[MAXD];
    double last_lp[MAXD];
    for (int d = 0; d < nd; ++d) {
        last[d] = 0xFFFFFFFFu;
        last_lp[d] = 0.0;
    }
    bool bad = false;
    double acc = 0.0;
    const int ngrp = (T + 3) >> 2;
    for (int grp = 0; grp < ngrp; ++grp) {
        uint32_t w[MAXD];
        for (int d = 0; d < nd; ++d) w[d] = ll_load4(P.bins + tile_offset(nd, ntile, d, grp, s));
        for (int j = 0; j < 4; ++j) {
            const int c = grp * 4 + j;
            if (c == 0 || c >= T) continue;
            for (int d = 0; d < nd; ++d) {
                uint32_t b = ((w[d] >> (8 * j)) & 0xFFu) - 1u;
                if (b >= (uint32_t)M.dyn[d].r) {
                    bad = true;
                    b = 0;
                }
                x[M.dyn_t1[d]] = (uint8_t)b;
            }
            for (int d = 0; d < nd; ++d) {
                const uint32_t o = ll_column(M.dyn[d], x) + x[M.dyn_t1[d]];
                if (o != last[d]) {   // bins mostly hold from one second to the next: gather only when the slot changes
                    last[d] = o;
                    last_lp[d] = ldg64(M.logp_trans + o);
                }
                acc = dadd(acc, last_lp[d]);
            }
            for (int d = 0; d < nd; ++d) x[M.dyn_t[d]] = x[M.dyn_t1[d]];
        }
    }
    if (bad) ll_flag(P.status, LL_BAD_BIN);
    return acc;
}

// Whole track s: initial term, column-0 check, transition term on the branch `frozen` selects.
template <class Cnt>
EMB_HD void loglik_track(const DevModel& M, const LoglikParams& P, int64_t s, bool frozen, Cnt cnt) {
    uint8_t x[MAXX];
    for (int i = 0; i < MAXX; ++i) x[i] = 0;
    const double init = loglik_initial_one(M, M.logp_init, P, s, x);
    if (P.initial) P.initial[s] = init;
    loglik_check_col0(M, P, s, x);
    if (!P.transition) return;
    for (int d = 0; d < M.n_dyn; ++d) x[M.dyn_t1[d]] = x[M.dyn_t[d]];
    P.transition[s] = frozen ? loglik_transition_frozen(M, P, s, x, cnt) : loglik_transition_step(M, P, s, x);
}

// counters per track of the frozen branch: sum of r over the dynamic variables
EMB_HD int loglik_counters(const DevModel& M) {
    int k = 0;
    for (int d = 0; d < M.n_dyn; ++d) k += M.dyn[d].r;
    return k;
}

}  // namespace emb
