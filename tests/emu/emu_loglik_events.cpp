// tests/emu/emu_loglik_events.cpp -- TEST-ONLY host emulation of the event-list scoring (emb_loglik_events.cuh).
//
// The __host__ __device__ per-track routine of k_loglik_events runs here on the CPU, one loop iteration per CUDA thread.
// tests/test_loglik_events.py builds it together with emu_loglik.cpp (model loading, the dense scoring it is compared with) into
// one library; NOT part of libemb200.so.
#include <cstdint>
#include <string>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_loglik_events.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_model.h"
#include "../../include/emb200.h"

using namespace emb;

static thread_local std::string g_err;

extern "C" {

const char* lle_last_error() { return g_err.c_str(); }

// emb_loglik_track_events (packed = 0, rows: emb_event) or emb_loglik_track_events_packed (packed = 1, rows: words + dts) on host
// buffers; the host-side refusals of the C ABI are the library's and are tested there
int lle_loglik_events(void* h, int64_t n, int32_t T, const int8_t* init_bins, const void* rows, const uint8_t* dts,
                      const int64_t* offsets, int32_t packed, int32_t correct_dbn, double* initial, double* transition) {
    const HostModel& H = *static_cast<HostModel*>(h);
    DevModel D = H.dev;
    D.logp_init = H.logp_initial.data();
    D.logp_trans = H.logp_transition.data();
    if (correct_dbn) D.fast = 0;
    int32_t status = 0;
    LoglikParams P{};
    P.n = n;
    P.T = T;
    P.init_bins = init_bins;
    P.initial = initial;
    P.transition = transition;
    P.status = &status;
    const EventRows R{offsets, static_cast<const uint32_t*>(rows), dts};
    int8_t dyn_of[MAXV];
    for (int v = 0; v < MAXV; ++v) dyn_of[v] = (int8_t)ll_dyn_of(D, v);
    std::vector<uint32_t> cnt((size_t)loglik_counters(D) + 1);
    auto c = [&](int k) -> uint32_t& { return cnt[(size_t)k]; };
    for (int64_t s = 0; s < n; ++s) {
        if (packed) loglik_track_events<true>(D, P, R, dyn_of, s, D.fast != 0, c);
        else loglik_track_events<false>(D, P, R, dyn_of, s, D.fast != 0, c);
    }
    return status;   // the LL_* bits; tests/test_loglik_events.py maps them to the library's messages
}

}  // extern "C"
