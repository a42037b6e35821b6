// tests/emu/emu_events_expand.cpp -- TEST-ONLY host emulation of the event-list expansion (emb_events_expand.cuh).
//
// The __host__ __device__ per-track routines of k_events_expand_count / k_events_expand run here on the CPU, one loop iteration
// per track, with a warp of one lane (ExpandLanes).  tests/test_events_expand.py builds it together with emu_loglik.cpp (model
// loading) into one library; NOT part of libemb200.so.
#include <cstdint>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_events_expand.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_model.h"

using namespace emb;

extern "C" {

// Both passes of emb_track_events_expand (packed = 0, rows: emb_event) or emb_track_events_expand_packed (packed = 1, rows:
// words + dts) on host buffers.  vars (0-based) / mul / div: the resolved control columns.  ctl_offsets[n+1] is always filled;
// controls (nullable) must hold ctl_offsets[n] rows, samples (nullable) n * T * n_initial doubles.  Returns the LL_* status bits.
int ee_expand(void* h, int64_t n, int32_t T, const double* init_values, const void* rows, const uint8_t* dts, const int64_t* offsets,
              int32_t packed, int32_t n_cols, const int32_t* vars, const double* mul, const double* div, double* samples,
              double* controls, int64_t* ctl_offsets) {
    const HostModel& H = *static_cast<HostModel*>(h);
    DevModel D = H.dev;
    D.edges = H.edges.data();
    int32_t status = 0;
    ExpandParams P{};
    P.n = n;
    P.T = T;
    P.n_cols = n_cols;
    P.init_values = init_values;
    P.status = &status;
    for (int j = 0; j < n_cols; ++j) {
        P.vars[j] = vars[j];
        P.mul[j] = mul[j];
        P.div[j] = div[j];
    }
    const EventRows R{offsets, static_cast<const uint32_t*>(rows), dts};
    const ExpandLanes L{0};
    std::vector<uint32_t> counts((size_t)n + 1);
    P.counts = counts.data();
    for (int64_t s = 0; s < n; ++s)
        counts[(size_t)s] = packed ? events_expand_count<true>(D, P, R, s, L) : events_expand_count<false>(D, P, R, s, L);
    ctl_offsets[0] = 0;
    for (int64_t s = 0; s < n; ++s) ctl_offsets[s + 1] = ctl_offsets[s] + counts[(size_t)s];
    if (status) return status;
    std::vector<long long> off((size_t)n + 1);
    for (int64_t s = 0; s <= n; ++s) off[(size_t)s] = ctl_offsets[s];
    P.ctl_offsets = off.data();
    P.controls = controls;
    P.samples = samples;
    ExpandShared S;
    for (int64_t s = 0; s < n; ++s) {
        if (packed) events_expand_track<true>(D, P, R, s, L, S);
        else events_expand_track<false>(D, P, R, s, L, S);
    }
    return status;   // tests/test_events_expand.py maps the bits to the library's messages
}

}  // extern "C"
