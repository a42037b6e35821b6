// tests/emu/emu.cpp -- TEST-ONLY host emulation of the device sampling routines.
//
// emb_device.cuh is written __host__ __device__; this file instantiates the *same* per-sample code
// on the CPU (one loop iteration per CUDA thread) so the `-m "not gpu"` test-suite can check the
// device logic against the oracle without a GPU.  It is NOT part of libemb200.so, is not reachable
// from the C ABI, and is never used by bench.py or the product path.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_fast.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_initial.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_integrate.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_model.h"
#include "../../include/emb200.h"

using namespace emb;

static thread_local std::string g_err;
static int g_use_fast = 0, g_last_fast = 0;

struct HostHist {
    unsigned long long* hi;
    unsigned long long* ht;
    void operator()(int which, int idx, int bin) const {
        unsigned long long* h = which ? ht : hi;
        if (h) h[idx * HIST_STRIDE + bin] += 1;
    }
};

extern "C" {

const char* emu_last_error() { return g_err.c_str(); }
void emu_use_fast(int on) { g_use_fast = on; }
int emu_last_fast() { return g_last_fast; }

int emu_model_load(const char* path, int overwrite, const int32_t* idx, int32_t n_idx, void** out) {
    try {
        *out = load_model_file(path, overwrite != 0, idx, idx ? n_idx : 0);
        return 0;
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
}
void emu_model_free(void* h) { delete static_cast<HostModel*>(h); }

int emu_set_prior(void* h, int which, int kind, double value) {
    HostModel& H = *static_cast<HostModel*>(h);
    try {
        (which ? H.prior_transition : H.prior_initial) = PriorSpec{kind, value};
        H.pack();
        return 0;
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
}

static DevModel host_dev(const HostModel& H) {
    DevModel D = H.dev;
    D.thr_init = H.thr_initial.data();
    D.thr_trans = H.thr_transition.data();
    D.edges = H.edges.data();
    D.dd32 = H.dd32.data();
    return D;
}

int emu_sample_initial(void* h, uint64_t seed, uint64_t first, int64_t n, const emb_sample_opts* o, int8_t* bins,
                       double* values, uint16_t* attempts) {
    const HostModel& H = *static_cast<HostModel*>(h);
    SampleParams P;
    try {
        fill_params(H, seed, first, n, 0, *o, P);
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
    P.start_ps = o->start_per_sample;      // host memory: the emulation runs the device code on the host
    P.start_stride = n;
    const DevModel D = host_dev(H);
    int status = 0;
    g_last_fast = 0;
    if (g_use_fast && initial_fast_ok(D, P)) {
        InitStrides st;
        fill_init_strides(D, (int)H.thr_initial.size(), 0, st);
        InitCalls ic;
        fill_init_calls(P, D.n_initial, ic);
        bool done = false;
#define EMB_X(NV_)                                                                                      \
    if (!done && D.n_initial == (NV_)) {                                                                \
        for (int64_t s0 = 0; s0 < n; s0 += INIT_SPT) {                                                  \
            if (values) initial_fast4<NV_, true, double, false>(D, P, st, ic, D.thr_init, D.dd32 + 4 * D.ddi_off[0], s0, bins, values, attempts); \
            else if (first & 3) initial_fast4<NV_, false, double, false>(D, P, st, ic, D.thr_init, D.dd32 + 4 * D.ddi_off[0], s0, bins, values, attempts); \
            else initial_fast4<NV_, false, double, true>(D, P, st, ic, D.thr_init, D.dd32 + 4 * D.ddi_off[0], s0, bins, values, attempts);    \
        }                                                                                               \
        done = true;                                                                                    \
    }
        EMB_INIT_SHAPES(EMB_X)
#undef EMB_X
        if (done) {
            g_last_fast = 1;
            return 0;
        }
    }
    for (int64_t s = 0; s < n; ++s) {
        uint8_t x[MAXX];
        double vals[MAXV];
        int attempt = sample_initial(D, P, P.first_sample + (uint64_t)s, x, vals);
        if (attempt < 0) {
            status = attempt == -2 ? 2 : 1;
            attempt = P.max_attempts;
        }
        if (attempts) attempts[s] = (uint16_t)(attempt + 1);
        for (int i = 0; i < D.n_initial; ++i) {
            if (bins) bins[(int64_t)i * n + s] = (int8_t)(x[i] + 1);
            if (values) values[(int64_t)i * n + s] = vals[i];
        }
    }
    if (status == 2) g_err = "Attempt to preset a dependent variable (or a preset bin out of range) in start_per_sample";
    return status == 2 ? EMB_E_ARG : status ? EMB_E_REJECT : 0;
}

int emu_sample_tracks(void* h, uint64_t seed, uint64_t first, int64_t n, int32_t T, const emb_sample_opts* o,
                      const emb_track_out* out) {
    const HostModel& H = *static_cast<HostModel*>(h);
    SampleParams P;
    try {
        fill_params(H, seed, first, n, T, *o, P);
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
    DevModel D = host_dev(H);
    if (o->correct_dbn) D.fast = 0;
    int32_t status = 0;
    TrackOut O{};
    O.bins = out->bins;
    O.values = out->values;
    O.init_bins = out->init_bins;
    O.init_values = out->init_values;
    O.attempts = out->attempts;
    O.hist_initial = out->hist_initial;
    O.hist_transition = out->hist_transition;
    O.status = &status;
    HostHist hh{out->hist_initial, out->hist_transition};
    bool done = false;
    if (g_use_fast) {
        const uint32_t rs = fast_shape_of(D);
        const bool fast = D.fast != 0;
        static FastShared S;
        if (rs) fast_fill_shared(D, S, 0, 1);   // only a fast shape fits FastShared (FAST_MAX_EDGES), as on the device
#define EMB_X(RS_, NG_, FAST_, ORD_)                                                   \
    if (!done && rs == (RS_) && D.n_gated == (NG_) && fast == (FAST_) && order_code(D) == (ORD_)) { \
        static CallTable<NG_> U;                                                      \
        for (int64_t s = 0; s < n; ++s) {                                             \
            if (s == P.s_end || s == 0) { P.s_begin = s; P.s_end = next_segment(P.first_sample, s, n); } \
            track_fast<RS_, NG_, FAST_, true, 0, ORD_>(D, P, O, s, true, S, U, 0, 1, hh); \
        }                                                                             \
        done = true;                                                                   \
    }
        EMB_FAST_SHAPES(EMB_X)
#undef EMB_X
    }
    g_last_fast = done ? 1 : 0;
    if (!done)
        for (int64_t s = 0; s < n; ++s) track_generic(D, P, O, s, hh);
    return status ? EMB_E_REJECT : 0;
}

// host emulation of emb_sample_track_events: pass 1 counts, prefix sum, pass 2 writes (same device code)
int emu_sample_track_events(void* h, uint64_t seed, uint64_t first, int64_t n, int32_t T, const emb_sample_opts* o,
                            int64_t capacity, emb_event* events, int64_t* offsets, int64_t* total_rows) {
    const HostModel& H = *static_cast<HostModel*>(h);
    SampleParams P;
    try {
        fill_params(H, seed, first, n, T, *o, P);
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
    DevModel D = host_dev(H);
    if (o->correct_dbn) D.fast = 0;
    int32_t status = 0;
    std::vector<uint32_t> counts((size_t)n);
    std::vector<long long> off((size_t)n + 1);
    HostHist hh{nullptr, nullptr};
    static FastShared S;
    const uint32_t rs = g_use_fast ? fast_shape_of(D) : 0;
    if (rs) fast_fill_shared(D, S, 0, 1);       // only a fast shape fits FastShared (FAST_MAX_EDGES), as on the device
    const bool fast = D.fast != 0;
    int max_bins = 0;
    for (int g = 0; g < D.n_gated; ++g) max_bins = std::max(max_bins, (int)D.init[D.gated_var[g]].r);
    EventFormat fm{};
    if (!event_format_for(D.n_gated, max_bins, T, fm)) return EMB_E_LIMIT;
    std::vector<uint32_t> words;       // the write pass produces packed rows; they are expanded to emb_event rows below
    std::vector<uint8_t> dts;
    for (int pass = 1; pass <= 2; ++pass) {
        TrackOut O{};
        O.status = &status;
        O.ev_gord_bits = fm.gord_bits;
        O.ev_dt_bytes = fm.dt_bytes;
        if (pass == 1) O.ev_counts = counts.data();
        else {
            words.assign((size_t)off[(size_t)n] + 1, 0u);
            dts.assign(((size_t)off[(size_t)n] + 1) * (size_t)fm.dt_bytes, 0);
            O.ev_offsets = off.data();
            O.ev_words = words.data();
            O.ev_dts = dts.data();
        }
        bool done = false;
#define EMB_X(RS_, NG_, FAST_, ORD_)                                                                    \
    if (!done && rs == (RS_) && D.n_gated == (NG_) && fast == (FAST_) && order_code(D) == (ORD_)) {     \
        static CallTable<NG_> U;                                                                        \
        for (int64_t s = 0; s < n; ++s) {                                                               \
            if (s == P.s_end || s == 0) { P.s_begin = s; P.s_end = next_segment(P.first_sample, s, n); } \
            if (pass == 1) track_fast<RS_, NG_, FAST_, false, 1, ORD_>(D, P, O, s, true, S, U, 0, 1, hh); \
            else track_fast<RS_, NG_, FAST_, false, 2, ORD_>(D, P, O, s, true, S, U, 0, 1, hh);           \
        }                                                                                               \
        done = true;                                                                                    \
    }
        EMB_FAST_SHAPES(EMB_X)
#undef EMB_X
        g_last_fast = done ? 1 : 0;
        if (!done)
            for (int64_t s = 0; s < n; ++s) track_generic(D, P, O, s, hh);
        if (pass == 1) {
            long long acc = 0;
            for (int64_t s = 0; s < n; ++s) {
                off[(size_t)s] = acc;
                acc += counts[(size_t)s];
            }
            off[(size_t)n] = acc;
            for (int64_t s = 0; s <= n; ++s) offsets[s] = off[(size_t)s];
            *total_rows = acc;
            if (acc > capacity) return EMB_E_LIMIT;
        }
    }
    for (long long i = 0; i < off[(size_t)n]; ++i) {
        const uint32_t dt_lo = fm.dt_bytes == 1 ? dts[(size_t)i] : reinterpret_cast<const uint16_t*>(dts.data())[i];
        const uint2 row = expand_event(D, words[(size_t)i], dt_lo, fm);
        std::memcpy(&events[i], &row, 8);
    }
    return status ? EMB_E_REJECT : 0;
}

// host emulation of emb_terminal_propagate (same per-chain code as k_terminal_chains); models = 10 HostModel* in
// TermParams::m order, geo = host doubles
int emu_terminal_propagate(void** models, uint64_t seed, uint64_t first, int64_t n, const double* geo, int64_t geo_stride,
                           const int32_t* geo_rows, double tmax_s, const emb_dyn_limits* limits, int32_t max_attempts,
                           float* traj, int16_t* len) {
    TermParams P;
    std::memset(&P, 0, sizeof(P));
    P.seed = seed;
    P.first_sample = first;
    P.n = n;
    P.tmax_s = tmax_s;
    term_round_keys(P.seed, P.rk);
    P.tmax = (int32_t)tmax_s;
    P.max_attempts = max_attempts > 0 ? max_attempts : 65535;
    P.geo = geo;
    P.geo_stride = geo_stride;
    for (int k = 0; k < 12; ++k) P.geo_row[k] = geo_rows[k];
    for (int a = 0; a < 2; ++a)
        P.lim[a] = TermLimits{limits[a].minVel_ft_s, limits[a].maxVel_ft_s, limits[a].maxTurnRate_deg_s,
                              limits[a].maxAltitude_ft, limits[a].maxVertRate_ft_s};
    std::vector<double> cuts((size_t)TERM_NMODELS * TERM_NCUT * TERM_CUT_MAX);
    P.cuts = cuts.data();
    try {
        for (int k = 0; k < TERM_NMODELS; ++k) {
            const HostModel& H = *static_cast<HostModel*>(models[k]);
            make_term_model(H, P.lim[k < 4 ? 0 : 1], P.m[k], cuts.data() + (size_t)k * TERM_NCUT * TERM_CUT_MAX);
            P.m[k].thr = H.thr_transition.data();
            P.m[k].edges = H.edges.data();
        }
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
    int32_t status = 0;
    TermOut O{traj, len, &status};
    for (int chain = 0; chain < 4; ++chain)
        for (int64_t s = 0; s < n; ++s) terminal_chain(P, O, s, chain);
    if (status & 2) return EMB_E_ARG;
    return (status & 1) ? EMB_E_REJECT : 0;
}

// discretize_bayes.m:14-22 against cutpoints_initial{i} (em_read.m:128-136), 0-based, straight from the model's boundaries
static int ref_discretize(const HostModel& H, int i, double x) {
    const int r = H.r_initial[i];
    const auto& e = H.boundaries[i];
    int b = 0;
    for (int j = 1; j < r; ++j) b += x >= (e.empty() ? (double)(j + 1) : e[(size_t)j]) ? 1 : 0;
    return b;
}

// bearing and distance cells of n points: cells_pc / cells_d2 = term_cell on the pseudo-angle and squared-norm tables the chain
// kernel uses, cells_ref / cells_dref = the reference's own route, discretize_bayes(wrapTo360(atan2d(y, x))) and
// discretize_bayes(norm([x y])) (createEncounter.m:277, :293); near[2] = dist_max_sq, quarter_sq
int emu_bearing_cells(void* model, int64_t n, const double* x, const double* y, int32_t* cells_pc, int32_t* cells_ref,
                      int32_t* cells_d2, int32_t* cells_dref, double* near) {
    const HostModel& H = *static_cast<HostModel*>(model);
    TermModel M;
    std::vector<double> cuts((size_t)TERM_NCUT * TERM_CUT_MAX);
    try {
        make_term_model(H, TermLimits{0.0, 1e9, 3.0, 1e9, 1e9}, M, cuts.data());
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
    for (int64_t i = 0; i < n; ++i) {
        cells_pc[i] = term_cell(cuts.data() + TC_BEAR * TERM_CUT_MAX, pseudo_angle(x[i], y[i]));
        cells_ref[i] = ref_discretize(H, M.i_bear, heading_of(y[i], x[i]));
        if (cells_d2) cells_d2[i] = term_cell(cuts.data() + TC_DIST2 * TERM_CUT_MAX, dadd(dmul(x[i], x[i]), dmul(y[i], y[i])));
        if (cells_dref) cells_dref[i] = ref_discretize(H, M.i_dist, norm2(x[i], y[i]));
    }
    if (near) {
        near[0] = M.dist_max_sq;
        near[1] = M.quarter_sq;
    }
    return 0;
}

// sind/cosd and the constant-divisor division of the chain kernel, for comparison with libm / IEEE division
void emu_sincosd(int64_t n, const double* x, double* s, double* c) {
    for (int64_t i = 0; i < n; ++i) sincosd(x[i], s[i], c[i]);
}
void emu_div_const(int64_t n, const double* a, double* by_ft, double* by_100) {
    for (int64_t i = 0; i < n; ++i) {
        by_ft[i] = div_const(a[i], TERM_FT_PER_NM, TERM_NM_PER_FT);
        by_100[i] = div_const(a[i], 100.0, 0.01);
    }
}

// host emulation of emb_tracks_integrate (same per-track code as k_tracks_integrate); g_* = tile ordinals
int emu_tracks_integrate(int64_t n, int32_t T, int32_t i_alt, int32_t i_speed, int32_t g_acc, int32_t g_vr, int32_t g_turn, int32_t n_tv,
                         double ur_speed, double ur_vertrate, double ur_heading, double min_speed, double max_speed,
                         const double* init_values, const float* values, float* xyz, uint8_t* is_good) {
    IntegrateParams P;
    std::memset(&P, 0, sizeof(P));
    P.n = n; P.T = T; P.i_alt = i_alt; P.i_speed = i_speed; P.g_acc = g_acc; P.g_vr = g_vr; P.g_turn = g_turn; P.n_tv = n_tv;
    P.ur_speed = ur_speed; P.ur_vertrate = ur_vertrate; P.ur_heading = ur_heading;
    P.min_speed = min_speed; P.max_speed = max_speed;
    P.init_values = init_values; P.values = values; P.xyz = xyz; P.is_good = is_good;
    for (int64_t s = 0; s < n; ++s) integrate_track(P, s);
    return 0;
}

// host emulation of emb_terminal_screen (same per-encounter code as k_terminal_screen)
int emu_terminal_screen(const float* traj, const int16_t* len, int64_t n, double tmax_s, double thres_dist_ft,
                        double thres_altlow_ft, double* hmd, double* vmd, int16_t* tcpa, int16_t* enc_time, uint8_t* runway) {
    ScreenParams P;
    std::memset(&P, 0, sizeof(P));
    P.n = n; P.tmax = (int32_t)tmax_s; P.thres_dist_ft = thres_dist_ft; P.thres_altlow_ft = thres_altlow_ft;
    P.traj = traj; P.len = len; P.hmd_ft = hmd; P.vmd_ft = vmd; P.tcpa = tcpa; P.enc_time_s = enc_time; P.runway = runway;
    for (int64_t s = 0; s < n; ++s) screen_encounter(P, s);
    return 0;
}

}  // extern "C"
