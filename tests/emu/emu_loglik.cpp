// tests/emu/emu_loglik.cpp -- TEST-ONLY host emulation of the log-likelihood routines (emb_loglik.cuh).
//
// Like emu.cpp for the samplers: the __host__ __device__ scoring code of k_loglik_initial / k_loglik_tracks runs here on the
// CPU, one loop iteration per CUDA thread, so the `-m "not gpu"` suite can check it against oracle/loglik.py and the GPU suite
// can check the device bit for bit against it.  Built on its own by tests/test_loglik.py; NOT part of libemb200.so.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_loglik.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_model.h"
#include "../../include/emb200.h"

using namespace emb;

static thread_local std::string g_err;

static DevModel host_dev(const HostModel& H) {
    DevModel D = H.dev;
    D.thr_init = H.thr_initial.data();
    D.thr_trans = H.thr_transition.data();
    D.edges = H.edges.data();
    D.dd32 = H.dd32.data();
    D.logp_init = H.logp_initial.data();
    D.logp_trans = H.logp_transition.data();
    return D;
}

static int loglik_status(int32_t status) {
    if (status & LL_BAD_BIN) g_err = "loglik: a bin is outside 1..r of its variable";
    else if (status & LL_BAD_COL0) g_err = "loglik: column 0 of the track bins differs from init_bins of the dynamic variables";
    return status ? EMB_E_ARG : 0;
}

extern "C" {

const char* ll_last_error() { return g_err.c_str(); }

int ll_model_load(const char* path, int overwrite, const int32_t* idx, int32_t n_idx, void** out) {
    try {
        *out = load_model_file(path, overwrite != 0, idx, idx ? n_idx : 0);
        return 0;
    } catch (const Error& e) {
        g_err = e.msg;
        return e.code;
    }
}
void ll_model_free(void* h) { delete static_cast<HostModel*>(h); }

int ll_set_prior(void* h, int which, int kind, double value) {
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

// the packed log tables (HostModel::logp_*), which = 0 initial / 1 transition; returns their length
int64_t ll_model_get_logp(void* h, int which, double* buf, int64_t cap) {
    const HostModel& H = *static_cast<HostModel*>(h);
    const auto& v = which ? H.logp_transition : H.logp_initial;
    if (buf) std::memcpy(buf, v.data(), sizeof(double) * (size_t)std::min<int64_t>(cap, (int64_t)v.size()));
    return (int64_t)v.size();
}

// emb_loglik_initial on host buffers (same per-sample code as k_loglik_initial)
int ll_loglik_initial(void* h, int64_t n, const int8_t* bins, double* total, double* per_var) {
    const HostModel& H = *static_cast<HostModel*>(h);
    const DevModel D = host_dev(H);
    int32_t status = 0;
    LoglikParams P{};
    P.n = n;
    P.init_bins = bins;
    P.initial = total;
    P.per_var = per_var;
    P.status = &status;
    uint8_t x[MAXV];
    for (int64_t s = 0; s < n; ++s) total[s] = loglik_initial_one(D, D.logp_init, P, s, x);
    return loglik_status(status);
}

// emb_loglik_tracks on host buffers (same per-track code as k_loglik_tracks)
int ll_loglik_tracks(void* h, int64_t n, int32_t T, const int8_t* init_bins, const int8_t* bins, int32_t correct_dbn,
                     double* initial, double* transition) {
    const HostModel& H = *static_cast<HostModel*>(h);
    if (!H.has_transition || H.temporal_map.empty()) {
        g_err = "dynvar:empty: model has no transition network";
        return EMB_E_ARG;
    }
    DevModel D = host_dev(H);
    if (correct_dbn) D.fast = 0;
    int32_t status = 0;
    LoglikParams P{};
    P.n = n;
    P.T = T;
    P.init_bins = init_bins;
    P.bins = bins;
    P.initial = initial;
    P.transition = transition;
    P.status = &status;
    std::vector<uint32_t> cnt((size_t)loglik_counters(D) + 1);
    for (int64_t s = 0; s < n; ++s) loglik_track(D, P, s, D.fast != 0, [&](int k) -> uint32_t& { return cnt[(size_t)k]; });
    return loglik_status(status);
}

}  // extern "C"
