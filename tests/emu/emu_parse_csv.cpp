// tests/emu/emu_parse_csv.cpp -- TEST-ONLY host emulation of the decimal table parser (emb_parse.cuh) and the CSV formatter of
// sample2track (emb_format.cuh: format_csv_track).
//
// The __host__ __device__ per-line routines of k_parse_lines / k_parse_values and the per-track routine of
// k_format_csv[_count] run here on the CPU, one loop iteration per line or track, with a warp of one lane (ExpandLanes).  Line
// discovery (k_parse_newline_count, k_parse_line_starts) is restated as a loop over the newlines, with the same starts array.
// tests/test_parse_csv.py builds it into a library of its own; NOT part of libemb200.so.
#include <cstdint>
#include <vector>

#include "../../em_model_manned_bayes_b200/csrc/emb_format.cuh"
#include "../../em_model_manned_bayes_b200/csrc/emb_parse.cuh"

using namespace emb;

extern "C" {

// emb_parse_table on host buffers: 0, -4 (EMB_E_ARG: *bad_line and *kind set) or -6 (EMB_E_LIMIT: *total_rows set)
int emu_parse_table(const char* text, int64_t bytes, int32_t cols, int64_t capacity_rows, double* values, int64_t* total_rows,
                    int64_t* bad_line, int32_t* kind) {
    *total_rows = 0;
    *bad_line = 0;
    *kind = -1;
    if (bytes == 0) return 0;
    std::vector<long long> starts(1, 0);
    for (int64_t i = 0; i < bytes; ++i)
        if (text[i] == '\n') starts.push_back(i + 1);
    starts.push_back(bytes + 1);
    const int64_t lines = (int64_t)starts.size() - 1;
    std::vector<uint32_t> rows((size_t)lines);
    std::vector<long long> row_of((size_t)lines + 1);
    unsigned long long err = PARSE_NO_ERROR;
    ParseParams P{};
    P.text = text;
    P.bytes = bytes;
    P.cols = cols;
    P.lines = lines;
    P.starts = starts.data();
    P.rows = rows.data();
    P.row_of = row_of.data();
    P.error = &err;
    for (int64_t i = 0; i < lines; ++i) parse_check_line(P, i);
    if (err != PARSE_NO_ERROR) {
        *bad_line = (int64_t)(err >> 2);
        *kind = (int32_t)(err & 3);
        return -4;
    }
    row_of[0] = 0;
    for (int64_t i = 0; i < lines; ++i) row_of[(size_t)i + 1] = row_of[(size_t)i] + rows[(size_t)i];
    *total_rows = row_of[(size_t)lines];
    if (*total_rows > capacity_rows) return -6;
    P.values = values;
    for (int64_t i = 0; i < lines; ++i) parse_values_line(P, i);
    return 0;
}

// "%.0f" of v[0..n) (floats widened to double) concatenated: offsets[n+1] always, text (nullable) must hold offsets[n] bytes.
// Returns 1 if a value is not finite.
int emu_format_f0(const float* v, int64_t n, char* text, int64_t* offsets) {
    int bad = 0;
    offsets[0] = 0;
    for (int64_t i = 0; i < n; ++i) {
        FmtCount c;
        bad |= !fmt_emit_f0(v[i], c);
        offsets[i + 1] = offsets[i] + c.n;
        if (text) {
            FmtWrite w{text + offsets[i]};
            fmt_emit_f0(v[i], w);
        }
    }
    return bad;
}

// both passes of emb_format_tracks_csv on host buffers: offsets[n+1] always; text (nullable) must hold offsets[n] bytes.
// Returns the FMT_* status bits.
int emu_format_tracks_csv(int64_t n, int32_t T, const float* xyz, const uint8_t* mask, char* text, int64_t* offsets) {
    int32_t status = 0;
    CsvParams P{};
    P.n = n;
    P.T = T;
    P.xyz = xyz;
    P.mask = mask;
    P.status = &status;
    const ExpandLanes L{0};
    std::vector<char> stage(FMT_STAGE_BYTES);
    offsets[0] = 0;
    for (int64_t s = 0; s < n; ++s) offsets[s + 1] = offsets[s] + format_csv_track<false>(P, s, L, nullptr);
    if (status || !text) return status;
    std::vector<long long> off((size_t)n + 1);
    for (int64_t s = 0; s <= n; ++s) off[(size_t)s] = offsets[s];
    P.offsets = off.data();
    P.text = text;
    for (int64_t s = 0; s < n; ++s) format_csv_track<true>(P, s, L, stage.data());
    return status;
}

}  // extern "C"
