// emb_model.h -- host-side model: parser (em_read.m semantics), derived fields, and the packer that
// turns count tables into word-space inverse-CDF threshold tables for the sm_100a kernels.
#pragma once
#include <cstdint>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "emb_device.cuh"
#include "emb_terminal.cuh"

struct emb_sample_opts;

namespace emb {

struct Error {
    int code;
    std::string msg;
};

struct PriorSpec {
    int kind = 0;       // EMB_PRIOR_*
    double value = 0.0;
};

// One conditional table: r x q counts, column-major (em_read.m:191-198).
struct Table {
    int32_t r = 0;
    int64_t q = 0;
    std::vector<int32_t> parents;  // 0-based variable ids in increasing order (asub2ind.m:13)
    std::vector<double> N;         // r*q
    bool present = false;
};

struct HostModel {
    // ---- as read (em_read.m:65-107) ----
    std::vector<std::string> labels_initial, labels_transition;
    int32_t n_initial = 0, n_transition = 0;
    std::vector<uint8_t> G_initial, G_transition;  // row-major [parent*n + child]
    std::vector<int32_t> r_initial, r_transition;
    std::vector<Table> T_initial;     // n_initial
    std::vector<Table> T_transition;  // n_transition (present only for the dynamic variables)
    std::vector<std::vector<double>> boundaries;  // n_initial; empty = '*'
    std::vector<double> resample_rates;
    bool has_boundaries = false, has_transition = false, temporal_map_given = false;
    // ---- derived (em_read.m:109-141, bn_sort.m) ----
    std::vector<int32_t> order_initial, order_transition;  // 0-based ids in topological order
    std::vector<std::pair<int32_t, int32_t>> temporal_map; // 0-based (var(t), var(t+1|t-1))
    std::vector<int32_t> zero_bins;                        // 1-based bin or 0
    std::vector<std::pair<double, double>> bounds_initial;
    bool is_dynvar_depend = false;                         // dbn_sample.m:55
    std::vector<int32_t> gated;                            // 0-based ids with rate > 0 or dynamic (value words)
    std::vector<int32_t> timevarying;                      // 0-based ids: dynamic(t) or gated
    // ---- priors ----
    PriorSpec prior_initial, prior_transition;
    // ---- packed (rebuilt by pack()) ----
    DevModel dev{};                    // metadata with null table pointers
    std::vector<uint32_t> thr_initial, thr_transition;
    // log(w_m / W) of the same columns, slot for slot (padding slots -inf): the scoring tables of emb_loglik.cuh
    std::vector<double> logp_initial, logp_transition;
    std::vector<double> edges;         // per variable: a[bin], w[bin] interleaved
    std::vector<float> dd32;           // per (gated ordinal, bin): {slope, base, s, c}
    uint64_t version = 0;

    // ---- device copies ----
    struct DeviceCopy {
        uint64_t version = ~0ull;
        uint32_t* thr_initial = nullptr;
        uint32_t* thr_transition = nullptr;
        double* edges = nullptr;
        float* dd32 = nullptr;
        // uploaded by the first scoring call on the device (emb_api.cpp: ensure_logp), dropped with the others on a repack
        bool logp_ok = false;
        double* logp_initial = nullptr;
        double* logp_transition = nullptr;
    };
    mutable std::mutex mu;
    mutable std::map<int, DeviceCopy> device_copies;

    void derive();   // throws Error
    void pack();     // throws Error
};

// throws Error
HostModel* load_model_file(const char* path, bool overwrite_zero_boundaries, const int32_t* idx_zero, int n_idx);

// Word-space thresholds of one column of weights w[0..r): fills col[0..rp) (see emb_device.cuh).
void pack_column(const double* w, int r, int rp, uint32_t* col);
// log(w_m / W) of the same column, W = sum(w) summed as select_random.m:17 does; a zero-total column gives bin 1 probability 1
// (log 0, every other bin -inf), as the sampler does; slots r .. rp-1 are -inf.
void logp_column(const double* w, int r, int rp, double* col);

// Validates `opts` (bn_sample.m:45-50 preset rule, driver options) and fills the kernel parameters; throws Error.
void fill_params(const HostModel& H, uint64_t seed, uint64_t first_sample, int64_t n, int32_t T,
                 const struct emb_sample_opts& opts, SampleParams& P);

// G = #{k in [0,2^32) : (k+0.5)*2^-32 < rate}  (resample_events.m:24 under the word->uniform map)
uint64_t gate_threshold(double rate);

// Terminal trajectory chains: checks the layout createEncounter.m:107-116 asserts and fills the per-chain model
// descriptor (table pointers left null; valid altitude/speed bins of :118-125 for `lim`) and, when `cuts` is given, its
// [TERM_NCUT][TERM_CUT_MAX] cutpoint tables (emb_terminal.cuh: term_cell); throws Error.
void make_term_model(const HostModel& H, const TermLimits& lim, TermModel& M, double* cuts = nullptr);
// @CorTerminalModel/getDynamicLimits.m:14-62; false if the aircraft type is unknown
bool named_dyn_limits(const char* ac_type, TermLimits& out);

}  // namespace emb
