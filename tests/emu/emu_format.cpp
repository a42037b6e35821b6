// tests/emu/emu_format.cpp -- TEST-ONLY host emulation of the em_sample text formatter (emb_format.cuh).
//
// The __host__ __device__ digit generation and per-track routines of k_format_{initial,transition}[_count] run here on the CPU, one
// loop iteration per track, with a warp of one lane (ExpandLanes).  tests/test_format.py builds it into a library of its own; NOT
// part of libemb200.so.
#include <cstdint>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_format.cuh"

using namespace emb;

extern "C" {

// "%g" of v[0..n) concatenated: offsets[n+1] always, text (nullable) must hold offsets[n] bytes.  Returns 1 if a value is not
// finite.
int emu_format_g(const double* v, int64_t n, char* text, int64_t* offsets) {
    int bad = 0;
    offsets[0] = 0;
    for (int64_t i = 0; i < n; ++i) {
        const G6 g = fmt_g6(v[i]);
        bad |= g.bad;
        FmtCount c;
        fmt_emit_g(g, c);
        offsets[i + 1] = offsets[i] + c.n;
        if (text) {
            FmtWrite w{text + offsets[i]};
            fmt_emit_g(g, w);
        }
    }
    return bad;
}

// Both passes of one text of emb_format_em_sample on host buffers: transition = 0 initial.txt (init_values [n_initial][n]),
// 1 transition.txt (values: the dense tiles, cols: tile ordinal of each dynamic variable).  offsets[n+1] always; text
// (nullable) must hold offsets[n] bytes.  Returns the FMT_* status bits.
int emu_format_em_sample(int64_t n, int32_t T, int64_t first_id, int32_t n_initial, int32_t n_dyn, int32_t n_tv, const int32_t* cols,
                         const double* init_values, const float* values, int32_t transition, char* text, int64_t* offsets) {
    int32_t status = 0;
    FormatParams P{};
    P.n = n;
    P.T = T;
    P.n_initial = n_initial;
    P.n_dyn = n_dyn;
    P.n_tv = n_tv;
    P.first_id = first_id;
    P.init_values = init_values;
    P.values = values;
    for (int j = 0; j < n_dyn; ++j) P.cols[j] = cols[j];
    P.status = &status;
    const ExpandLanes L{0};
    std::vector<char> stage(FMT_STAGE_BYTES);
    offsets[0] = 0;
    for (int64_t s = 0; s < n; ++s)
        offsets[s + 1] = offsets[s] + (transition ? format_track<true, false>(P, s, L, nullptr) : format_track<false, false>(P, s, L, nullptr));
    if (status || !text) return status;
    std::vector<long long> off((size_t)n + 1);
    for (int64_t s = 0; s <= n; ++s) off[(size_t)s] = offsets[s];
    P.offsets = off.data();
    P.text = text;
    for (int64_t s = 0; s < n; ++s) {
        if (transition) format_track<true, true>(P, s, L, stage.data());
        else format_track<false, true>(P, s, L, stage.data());
    }
    return status;
}

}  // extern "C"
