// emb_events_expand.cuh -- out_samples and the control rows of tracks given as event lists (the rows of
// emb_sample_track_events[_packed]): the per-track routines of k_events_expand_count / k_events_expand (emb_kernels.cu).
// __host__ __device__ like emb_loglik_events.cuh, so that tests/emu runs the same code on the CPU.
//
// The result is defined by reduction to the host statements (emb200.h: emb_track_events_expand):
//  - samples: events2samples.m:9-27 / model.py expand_events -- a row is visible from column sum(dt up to and including it)
//    on, the last row wins within a column, rows at column >= T change nothing, sum(dt) < T holds the last state;
//  - controls: events2controls.m:9-31 -- one row [t, y_1 .. y_k] per list row with dt > 0, t the seconds before the row and
//    y_j = (x[vars_j] * mul_j) / div_j of the state x before the row (two correctly rounded fp64 operations).
// Values pass through unchanged: an 8-byte row's fp32 value widened to fp64, a packed row's value from dedisc() exactly as
// PackedEventResult.decode computes it.
//
// Shape: one warp per track.  The warp reads the rows in chunks of 32, one row per lane (coalesced loads).  A warp scan of dt
// gives every row its column and the seconds before it; one ballot per initial variable gives, for every lane, the last lane
// below it that set the variable ("last writer"), so the state before any row is a shared-memory read.  Runs of columns with
// constant state are contiguous blocks of [T][n_initial] doubles, stored by the whole warp; control rows are staged in shared
// memory and stored as one contiguous block per chunk.  The host emulation runs the same code with a warp of one lane.
#pragma once
#include "emb_loglik_events.cuh"

namespace emb {

struct ExpandParams {
    int64_t n;
    int32_t T;
    int32_t n_cols;                   // control columns after t (1..MAXD)
    const double* init_values;        // [n_initial][n]
    double* samples;                  // [n][T][n_initial] or nullptr
    const long long* ctl_offsets;     // [n+1] control rows before each track (write pass)
    double* controls;                 // [total][1 + n_cols] or nullptr (write pass)
    uint32_t* counts;                 // [n] control rows of each track (count pass)
    int32_t* status;                  // LL_BAD_VAR / LL_BAD_BIN / LL_BAD_OFFSETS
    int32_t vars[MAXD];               // 0-based initial variable of each control column
    double mul[MAXD], div[MAXD];
};

EMB_HD double ddiv(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    volatile double r = a / b;
    return r;
#endif
}

EMB_HD int ee_top(uint32_t m) {   // highest set bit of m != 0
#if defined(__CUDA_ARCH__)
    return 31 - __clz(m);
#else
    return 31 - __builtin_clz(m);
#endif
}
EMB_HD int ee_low(uint32_t m) {   // lowest set bit of m != 0
#if defined(__CUDA_ARCH__)
    return __ffs(m) - 1;
#else
    return __builtin_ctz(m);
#endif
}
EMB_HD int ee_popc(uint32_t m) {
#if defined(__CUDA_ARCH__)
    return __popc(m);
#else
    return __builtin_popcount(m);
#endif
}

// The lanes that work on one track: a full warp on the device, one lane in the host emulation.
struct ExpandLanes {
    int lane;
    EMB_HD static int width() {
#if defined(__CUDA_ARCH__)
        return 32;
#else
        return 1;
#endif
    }
    EMB_HD uint32_t ballot(bool p) const {
#if defined(__CUDA_ARCH__)
        return __ballot_sync(0xFFFFFFFFu, p);
#else
        return p ? 1u : 0u;
#endif
    }
    EMB_HD int32_t scan(int32_t v) const {   // inclusive prefix sum over the lanes
#if defined(__CUDA_ARCH__)
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t y = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += y;
        }
#endif
        return v;
    }
    EMB_HD int32_t last(int32_t v) const {   // the value of the last lane
#if defined(__CUDA_ARCH__)
        return __shfl_sync(0xFFFFFFFFu, v, 31);
#else
        return v;
#endif
    }
    EMB_HD void sync() const {
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
    }
};

// shared memory of one warp
struct ExpandShared {
    double val[32];                   // value the lane's row sets
    int32_t col[32];                  // column the lane's row is visible from, saturated at T
    uint32_t mask[MAXV];              // lanes whose row sets initial variable i
    double x[MAXV];                   // state before the chunk
    double ctl[32 * (1 + MAXD)];      // the chunk's control rows
};

EMB_HD bool ee_offsets(const EventRows& R, int64_t n, int64_t s, int64_t& a, int64_t& e) {
    a = R.offsets[s];
    e = R.offsets[s + 1];
    if (a < 0 || e < a || e > R.offsets[n]) {
        e = a;
        return false;
    }
    return true;
}

// Count pass: control rows of track s (rows with dt > 0).  Reads the dt of every row.
template <bool PACKED>
EMB_HD uint32_t events_expand_count(const DevModel& M, const ExpandParams& P, const EventRows& R, int64_t s, const ExpandLanes& L) {
    const int W = ExpandLanes::width();
    int64_t a, e;
    if (!ee_offsets(R, P.n, s, a, e) && L.lane == 0) ll_flag(P.status, LL_BAD_OFFSETS);
    uint32_t rows = 0;
    for (int64_t base = a; base < e; base += W) {
        const int64_t row = base + L.lane;
        uint32_t dt = 0, bin;
        int v;
        if (row < e) ll_event_row<PACKED>(M, R, row, dt, v, bin);
        rows += (uint32_t)ee_popc(L.ballot(dt > 0));
    }
    return rows;
}

// Write pass: the samples of track s (P.samples) and its control rows from row P.ctl_offsets[s] on (P.controls).
template <bool PACKED>
EMB_HD void events_expand_track(const DevModel& M, const ExpandParams& P, const EventRows& R, int64_t s, const ExpandLanes& L,
                                ExpandShared& S) {
    const int W = ExpandLanes::width(), lane = L.lane, ni = M.n_initial, T = P.T, k = P.n_cols;
    int64_t a, e;
    int32_t bad = ee_offsets(R, P.n, s, a, e) ? 0 : LL_BAD_OFFSETS;
    for (int i = lane; i < ni; i += W) S.x[i] = P.init_values[(int64_t)i * P.n + s];
    L.sync();
    double* out = P.samples ? P.samples + (int64_t)s * T * ni : nullptr;
    const int i0 = lane % ni, istep = W % ni;
    // columns [c0, c1) of the samples with the state before the row of the lane whose lanes below are `below`
    auto fill = [&](int c0, int c1, uint32_t below) {
        double* dst = out + (int64_t)c0 * ni;
        const int count = (c1 - c0) * ni;
        int i = i0;
        for (int el = lane; el < count; el += W) {
            const uint32_t m = S.mask[i] & below;
            dst[el] = m ? S.val[ee_top(m)] : S.x[i];
            i += istep;
            if (i >= ni) i -= ni;
        }
    };
    const uint32_t below = (1u << lane) - 1u;
    int written = 0;                                        // columns [0, written) of the samples are stored
    int64_t t = 0;                                          // seconds before the chunk
    int64_t q = P.controls ? (int64_t)P.ctl_offsets[s] : 0; // next control row
    for (int64_t base = a; base < e; base += W) {
        const int64_t row = base + lane;
        uint32_t dt = 0, bin = 0;
        int v = -1;
        double val = 0.0;
        if (row < e) {
            ll_event_row<PACKED>(M, R, row, dt, v, bin);
            if (v == -2) {
                bad |= LL_BAD_VAR;
                v = -1;
            } else if (v >= 0 && PACKED) {
                if (bin - 1u >= (uint32_t)M.init[v].r) {   // the edge table of v has r pairs
                    bad |= LL_BAD_BIN;
                    v = -1;
                } else {
                    const uint32_t frac = ll_ldg32(R.words + row) & 0x7FFFFFu;
                    val = dedisc(M, v, (int)bin - 1, dmul(dadd((double)frac, 0.5), 1.1920928955078125e-07));
                }
            } else if (v >= 0) {
                const uint32_t bits = ll_ldg32(R.words + 2 * row + 1);
                float f;
#if defined(__CUDA_ARCH__)
                f = __uint_as_float(bits);
#else
                std::memcpy(&f, &bits, 4);
#endif
                val = (double)f;
            }
        }
        const int32_t incl = L.scan((int32_t)dt);
        const int64_t tc = t + incl;                        // the row is visible from column tc
        const int col = tc < T ? (int)tc : T;
        S.col[lane] = col;
        S.val[lane] = val;
        for (int i = 0; i < ni; ++i) {
            const uint32_t m = L.ballot(v == i);
            if (lane == 0) S.mask[i] = m;
        }
        L.sync();
        if (P.controls) {
            const uint32_t cm = L.ballot(dt > 0);
            if (dt > 0) {
                double* c = S.ctl + ee_popc(cm & below) * (1 + k);
                c[0] = (double)(tc - (int64_t)dt);
                for (int j = 0; j < k; ++j) {
                    const int i = P.vars[j];
                    const uint32_t m = S.mask[i] & below;
                    c[1 + j] = ddiv(dmul(m ? S.val[ee_top(m)] : S.x[i], P.mul[j]), P.div[j]);
                }
            }
            L.sync();
            const int count = ee_popc(cm) * (1 + k);
            double* dst = P.controls + q * (1 + k);
            for (int el = lane; el < count; el += W) dst[el] = S.ctl[el];
            q += ee_popc(cm);
        }
        if (out && written < T) {
            const int prev = lane ? S.col[lane - 1] : written;
            for (uint32_t starts = L.ballot(col > prev); starts; starts &= starts - 1u) {   // rows that open a new column
                const int r = ee_low(starts);
                fill(r ? S.col[r - 1] : written, S.col[r], (1u << r) - 1u);
            }
        }
        t += L.last(incl);
        written = S.col[W - 1];
        L.sync();
        for (int i = lane; i < ni; i += W)
            if (S.mask[i]) S.x[i] = S.val[ee_top(S.mask[i])];
        L.sync();
    }
    if (out && written < T) fill(written, T, 0u);
    if (bad) ll_flag(P.status, bad);
}

}  // namespace emb
