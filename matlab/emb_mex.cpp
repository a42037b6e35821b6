// emb_mex.cpp -- thin MEX gateway from MATLAB to the C ABI of libemb200.so (include/emb200.h).
//
// SOURCE ONLY: this image has no MATLAB (no mex.h), so the file is never compiled by build() and no
// test links it; it documents the binding a maintainer adds (see INTEGRATION.md):
//     mex -R2018a matlab/emb_mex.cpp -Iinclude -Lem_model_manned_bayes_b200 -lemb200
//
//   h    = emb_mex('load', parameters_filename, isOverwriteZeroBoundaries, idxZeroBoundaries)
//   h    = emb_mex('from_arrays', G_initial, r_initial, w_initial, G_transition, r_transition, w_transition, ...
//                  temporal_map, boundaries, resample_rates)
//          the object form (EncounterModel.m:5-70 properties; matlab/emb_handle.m): G_* logical n x n (G(parent, child)),
//          r_* n x 1, w_* the weight tables N{i} + alpha{i} of all variables back to back (each r_i x q_i, column-major,
//          variable order: em_read.m:191-198), temporal_map k x 2, boundaries 1 x n_initial cell, resample_rates n_initial x 1
//   s    = emb_mex('info', h)                       % struct mirroring emb_model_info (1-based ids)
//          emb_mex('set_prior', h, which, kind, value)
//   [bins, values, attempts] = emb_mex('sample_initial', h, seed, first, n, opts)
//   [out_inits, bins, values, attempts] = emb_mex('sample_tracks', h, seed, first, n, T, opts)
//   [out_inits, bins, values, hist_i, hist_t] = emb_mex('sample_tracks_multi', h, seed, first, n, T, opts, n_devices)
//          all GPUs of the box from one call (emb_sample_tracks_multi): bins / values are 1 x D cells of per-device tiles
//   [events, offsets, out_inits, attempts, init_bins, out_samples, ctl] = emb_mex('sample_events', h, seed, first, n, T, opts)
//          events: 4 x rows double [dt; var; value; bin], offsets: (n+1) x 1 (0-based first row of each track),
//          init_bins: n x n_initial int8 (the initial bins, what 'loglik_events' needs),
//          out_samples: n x 1 cell of n_initial x T (events2samples.m), ctl: n x 1 cell of the out_EME event matrices
//          [t, dh/60, deg2rad(dpsi), dv*1.68780972222222] (UncorEncounterModel.m:286-297) -- both computed on the GPU from
//          the same rows (emb_track_events_expand[_packed]), and only when requested
//   [traj, len] = emb_mex('terminal_propagate', hs, seed, first, geo, tmax_s, limits, opts)
//          hs: 1 x 10 uint64 handles {own_fwd(1:2), own_bck(1:2), int_fwd(1:3), int_bck(1:3)}; geo: n x 12 double
//          [own_intent own_distance own_bearing own_alt own_heading own_speed int_...]; limits: 5 x 2 double
//          [minVel; maxVel; maxTurnRate; maxAltitude; maxVertRate] per aircraft;
//          traj: n x (2*tmax+1) x 2 x 5 single (NaN = no state), len: n x 4 int16
//   s = emb_mex('terminal_screen', traj, len, tmax_s, thresDist_ft, thresAltLow_ft)   % traj/len as returned above
//          struct: hmd_ft, vmd_ft (n x 1 double), tcpa (n x 3 int16: tcpa_s, index_own, index_int), enc_time_s, runway (bits)
//   [xyz, is_good] = emb_mex('tracks_integrate', h, out_inits, values, T, iopts)    % sample2track.m:188-244
//          out_inits n x n_initial double and values 4 x 128 x n_tv x ceil(n/128) x ceil(T/4) single as returned by 'sample_tracks';
//          iopts: struct idx_altitude, idx_speed, idx_acceleration, idx_vertrate, idx_turnrate, ur_speed, ur_vertrate,
//          ur_heading, min_speed, max_speed;  xyz: n x (T+1) x 3 single, is_good: n x 1 uint8
//   [xyz, is_good, out_inits] = emb_mex('sample_tracks_xyz', h, seed, first, n, T, opts, iopts)
//          sampling and the loop of sample2track.m:188-244 in one kernel pass (no dense tiles); outputs as above
//   [initial, transition] = emb_mex('em_sample_text', h, seed, first, n, T, opts)   % em_sample.m:88-100 on the GPU
//          the rows of initial.txt and transition.txt (without header lines) as uint8 row vectors, ids first+1 .. first+n,
//          numbers as fprintf's "%g" prints them (emb_format_em_sample); matlab/em_sample_b200.m writes the files
//   [total, per_var] = emb_mex('loglik_initial', h, bins)              % log p of initial states (emb_loglik_initial)
//          bins: n x n_initial int8 (1-based); total n x 1, per_var n x n_initial double
//   [initial, transition] = emb_mex('loglik_tracks', h, init_bins, bins, T, correct_dbn)   % log p of tracks
//          init_bins: n x n_initial int8; bins: the tiled int8 array of 'sample_tracks'; initial, transition n x 1 double
//   [initial, transition] = emb_mex('loglik_events', h, init_bins, events, offsets, T, correct_dbn)   % log p of event lists
//          init_bins, events (4 x rows [dt; var; value; bin]) and offsets as 'sample_events' returns them; the bin row is
//          required (a 3-row out_events without bins is refused); equal to 'loglik_tracks' on the same tracks
//          emb_mex('free', h)
// opts: struct with optional fields start (1 x n_initial, 0/NaN = free), reject_mode, idx_v, idx_dh,
// idx_L, is_quantize500, layers (r_L x 2), box_lo, box_hi, max_attempts, device, start_per_sample (n x n_initial, 0/NaN = free:
// one `start` row per sample, the cell of @CorTerminalModel/InitStartTerminal.m as a matrix).
// Errors become mexErrMsgIdAndTxt with the reference's identifiers where the reference has one
// ('dynvar:empty', UncorEncounterModel.m:231-234; 'prior:notdbe', EncounterModel.m:200).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "emb200.h"
#include "mex.h"

namespace {

void fail(int rc) {
    const char* msg = emb_last_error();
    const char* id = "emb200:error";
    if (std::strstr(msg, "dynvar:empty")) id = "dynvar:empty";
    else if (std::strstr(msg, "prior:")) id = "prior:notdbe";
    else if (rc == EMB_E_CUDA) id = "emb200:cuda";
    else if (rc == EMB_E_REJECT) id = "emb200:reject";
    mexErrMsgIdAndTxt(id, "%s", msg);
}
#define CHECK(call) do { int rc__ = (call); if (rc__ != 0) fail(rc__); } while (0)

emb_model* handle(const mxArray* a) {
    if (!mxIsUint64(a) || mxGetNumberOfElements(a) != 1) mexErrMsgIdAndTxt("emb200:arg", "bad model handle");
    return reinterpret_cast<emb_model*>(*static_cast<uint64_t*>(mxGetData(a)));
}

double field_or(const mxArray* s, const char* name, double dflt) {
    const mxArray* f = s && mxIsStruct(s) ? mxGetField(s, 0, name) : nullptr;
    return f && !mxIsEmpty(f) ? mxGetScalar(f) : dflt;
}

// int8 [n_initial][n] copy of opts.start_per_sample (n x n_initial double, 0 / NaN = free), alive for the duration of the call
std::vector<int8_t> g_start_rows;

void fill_opts(const mxArray* s, int n_initial, emb_sample_opts* o) {
    emb_sample_opts_init(o);
    o->mem = EMB_MEM_HOST;
    o->device = (int)field_or(s, "device", -1);
    o->reject_mode = (int)field_or(s, "reject_mode", EMB_REJECT_NONE);
    o->idx_v = (int)field_or(s, "idx_v", 0);
    o->idx_dh = (int)field_or(s, "idx_dh", 0);
    o->idx_L = (int)field_or(s, "idx_L", 0);
    o->is_quantize500 = (int)field_or(s, "is_quantize500", 0);
    o->max_attempts = (int)field_or(s, "max_attempts", 0);
    if (!s || !mxIsStruct(s)) return;
    if (const mxArray* st = mxGetField(s, 0, "start")) {          // bn_sample.m:45: empty/NaN = free
        const double* p = mxGetPr(st);
        for (size_t i = 0; i < mxGetNumberOfElements(st) && (int)i < n_initial; ++i)
            o->start[i] = std::isnan(p[i]) ? 0 : (int32_t)p[i];
    }
    if (const mxArray* sp = mxGetField(s, 0, "start_per_sample")) {   // rows of InitStartTerminal.m, one per sample
        if (!mxIsEmpty(sp)) {
            const size_t cnt = mxGetNumberOfElements(sp);             // column-major n x n_initial == [n_initial][n]
            const double* p = mxGetPr(sp);
            g_start_rows.resize(cnt);
            for (size_t i = 0; i < cnt; ++i) g_start_rows[i] = std::isnan(p[i]) ? (int8_t)0 : (int8_t)p[i];
            o->start_per_sample = g_start_rows.data();
        }
    }
    if (const mxArray* ly = mxGetField(s, 0, "layers")) {         // UncorEncounterModel.m:259-263, r_L x 2 column-major
        const size_t r = mxGetM(ly);
        const double* p = mxGetPr(ly);
        o->n_layers = (int32_t)r;
        for (size_t k = 0; k < r && k < 8; ++k) { o->layers[k][0] = p[k]; o->layers[k][1] = p[r + k]; }
    }
    for (const char* nm : {"box_lo", "box_hi"})
        if (const mxArray* b = mxGetField(s, 0, nm)) {
            const double* p = mxGetPr(b);
            double* dst = nm[4] == 'l' ? o->box_lo : o->box_hi;
            for (size_t i = 0; i < mxGetNumberOfElements(b) && (int)i < n_initial; ++i) dst[i] = p[i];
        }
}

}  // namespace

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 1 || !mxIsChar(prhs[0])) mexErrMsgIdAndTxt("emb200:arg", "first argument must be a command string");
    char cmd[32];
    mxGetString(prhs[0], cmd, sizeof(cmd));
    const std::string c(cmd);

    if (c == "trim") {                                            // return the pooled per-call temporaries to the driver
        CHECK(emb_trim_device_memory(nrhs > 1 ? (int)mxGetScalar(prhs[1]) : -1));
        return;
    }
    if (c == "load") {                                            // replaces em_read.m:1-141
        char path[4096];
        mxGetString(prhs[1], path, sizeof(path));
        const int overwrite = nrhs > 2 ? (int)mxGetScalar(prhs[2]) : 0;
        std::vector<int32_t> idx;
        if (nrhs > 3)
            for (size_t i = 0; i < mxGetNumberOfElements(prhs[3]); ++i) idx.push_back((int32_t)mxGetPr(prhs[3])[i]);
        emb_model* m = nullptr;
        CHECK(emb_model_load(path, overwrite, idx.data(), (int32_t)idx.size(), &m));
        plhs[0] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
        *static_cast<uint64_t*>(mxGetData(plhs[0])) = reinterpret_cast<uint64_t>(m);
        return;
    }
    if (c == "from_arrays") {                                     // EncounterModel objects built without a file (EncounterModel.m:106-114)
        if (nrhs < 10) mexErrMsgIdAndTxt("emb200:arg", "from_arrays needs 9 arguments");
        auto as_i32 = [](const mxArray* a) {
            std::vector<int32_t> v(mxGetNumberOfElements(a));
            for (size_t i = 0; i < v.size(); ++i) v[i] = (int32_t)mxGetPr(a)[i];
            return v;
        };
        auto graph = [](const mxArray* a) {                       // MATLAB G(parent, child), column-major -> ABI G[parent * n + child]
            const size_t n = mxGetM(a);
            std::vector<uint8_t> g(n * n);
            const mxLogical* src = mxIsLogical(a) ? mxGetLogicals(a) : nullptr;
            for (size_t pa = 0; pa < n; ++pa)
                for (size_t ch = 0; ch < n; ++ch)
                    g[pa * n + ch] = (uint8_t)(src ? src[ch * n + pa] : mxGetPr(a)[ch * n + pa] != 0.0);
            return g;
        };
        const std::vector<uint8_t> Gi = graph(prhs[1]), Gt = graph(prhs[4]);
        const std::vector<int32_t> ri = as_i32(prhs[2]), rt = as_i32(prhs[5]);
        const int32_t n_initial = (int32_t)ri.size(), n_transition = (int32_t)rt.size();
        std::vector<int32_t> tmap(mxGetNumberOfElements(prhs[7]));
        const size_t k = mxGetM(prhs[7]);
        for (size_t r = 0; r < k; ++r) {                          // k x 2 column-major -> row-major pairs
            tmap[2 * r] = (int32_t)mxGetPr(prhs[7])[r];
            tmap[2 * r + 1] = (int32_t)mxGetPr(prhs[7])[k + r];
        }
        std::vector<double> bnd;
        std::vector<int32_t> bnd_len((size_t)n_initial, 0);
        for (int32_t i = 0; i < n_initial && (size_t)i < mxGetNumberOfElements(prhs[8]); ++i) {
            const mxArray* b = mxGetCell(prhs[8], i);
            const size_t m = b ? mxGetNumberOfElements(b) : 0;
            bnd_len[(size_t)i] = (int32_t)m;
            for (size_t q = 0; q < m; ++q) bnd.push_back(mxGetPr(b)[q]);
        }
        std::vector<double> rates((size_t)n_initial, 0.0);
        for (size_t i = 0; i < rates.size() && i < mxGetNumberOfElements(prhs[9]); ++i) rates[i] = mxGetPr(prhs[9])[i];
        emb_model* m = nullptr;
        CHECK(emb_model_from_arrays(n_initial, Gi.data(), ri.data(), mxGetPr(prhs[3]), (int64_t)mxGetNumberOfElements(prhs[3]),
                                    n_transition, n_transition ? Gt.data() : nullptr, n_transition ? rt.data() : nullptr,
                                    n_transition ? mxGetPr(prhs[6]) : nullptr, (int64_t)mxGetNumberOfElements(prhs[6]),
                                    tmap.data(), (int32_t)k, bnd.data(), bnd_len.data(), rates.data(), &m));
        plhs[0] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
        *static_cast<uint64_t*>(mxGetData(plhs[0])) = reinterpret_cast<uint64_t>(m);
        return;
    }
    if (c == "terminal_propagate") {                              // @CorTerminalModel/createEncounter.m:1-329 over a batch
        if (!mxIsUint64(prhs[1]) || mxGetNumberOfElements(prhs[1]) != 10) mexErrMsgIdAndTxt("emb200:arg", "need 10 model handles");
        const uint64_t* hs = static_cast<const uint64_t*>(mxGetData(prhs[1]));
        emb_terminal_models tm;
        for (int k = 0; k < 2; ++k) { tm.own_fwd[k] = reinterpret_cast<emb_model*>(hs[k]); tm.own_bck[k] = reinterpret_cast<emb_model*>(hs[2 + k]); }
        for (int k = 0; k < 3; ++k) { tm.int_fwd[k] = reinterpret_cast<emb_model*>(hs[4 + k]); tm.int_bck[k] = reinterpret_cast<emb_model*>(hs[7 + k]); }
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetM(prhs[4]);                // geo is n x 12 column-major == [12][n]
        const double tmax_s = mxGetScalar(prhs[5]);
        emb_dyn_limits lim[2];
        for (int a = 0; a < 2; ++a) {
            const double* p = mxGetPr(prhs[6]) + 5 * a;
            lim[a] = emb_dyn_limits{p[0], p[1], p[2], p[3], p[4]};
        }
        emb_sample_opts o;
        fill_opts(nrhs > 7 ? prhs[7] : nullptr, 0, &o);
        const int32_t rows[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
        const mwSize S = (mwSize)(2 * (int64_t)tmax_s + 1);
        const mwSize dt[4] = {(mwSize)n, S, 2, EMB_TRAJ_FIELDS};   // [field][aircraft][slot][n] == n x S x 2 x 5 column-major
        plhs[0] = mxCreateNumericArray(4, dt, mxSINGLE_CLASS, mxREAL);
        mxArray* len = mxCreateNumericMatrix(n, 4, mxINT16_CLASS, mxREAL);
        emb_traj_out out{(float*)mxGetData(plhs[0]), (int16_t*)mxGetData(len)};
        CHECK(emb_terminal_propagate(&tm, &rng, n, mxGetPr(prhs[4]), n, rows, tmax_s, lim, &o, &out));
        if (nlhs > 1) plhs[1] = len; else mxDestroyArray(len);
        return;
    }
    if (c == "terminal_screen") {                                 // CorTerminalModel.m:117-133, :187-210, track.m:88
        const int64_t n = (int64_t)mxGetM(prhs[2]);
        const char* names[] = {"hmd_ft", "vmd_ft", "tcpa", "enc_time_s", "runway"};
        plhs[0] = mxCreateStructMatrix(1, 1, 5, names);
        mxArray* hmd = mxCreateDoubleMatrix(n, 1, mxREAL);
        mxArray* vmd = mxCreateDoubleMatrix(n, 1, mxREAL);
        mxArray* tcpa = mxCreateNumericMatrix(n, 3, mxINT16_CLASS, mxREAL);
        mxArray* enc = mxCreateNumericMatrix(n, 1, mxINT16_CLASS, mxREAL);
        mxArray* rw = mxCreateNumericMatrix(n, 1, mxUINT8_CLASS, mxREAL);
        emb_sample_opts o;
        emb_sample_opts_init(&o);
        emb_screen_out so{mxGetPr(hmd), mxGetPr(vmd), (int16_t*)mxGetData(tcpa), (int16_t*)mxGetData(enc), (uint8_t*)mxGetData(rw)};
        CHECK(emb_terminal_screen((const float*)mxGetData(prhs[1]), (const int16_t*)mxGetData(prhs[2]), n, mxGetScalar(prhs[3]),
                                  mxGetScalar(prhs[4]), mxGetScalar(prhs[5]), &o, &so));
        mxSetField(plhs[0], 0, "hmd_ft", hmd); mxSetField(plhs[0], 0, "vmd_ft", vmd); mxSetField(plhs[0], 0, "tcpa", tcpa);
        mxSetField(plhs[0], 0, "enc_time_s", enc); mxSetField(plhs[0], 0, "runway", rw);
        return;
    }
    emb_model* m = handle(prhs[1]);
    emb_model_info info;
    CHECK(emb_model_get_info(m, &info));
    const int ni = info.n_initial;

    if (c == "free") {
        emb_model_free(m);
    } else if (c == "info") {
        const char* names[] = {"n_initial", "n_transition", "n_dyn", "is_dynvar_depend", "r_initial", "order_initial",
                               "temporal_map", "zero_bins", "resample_rates", "timevarying_vars"};
        plhs[0] = mxCreateStructMatrix(1, 1, 10, names);
        auto scalar = [&](const char* f, double v) { mxSetField(plhs[0], 0, f, mxCreateDoubleScalar(v)); };
        auto vec = [&](const char* f, int n, auto get) {
            mxArray* a = mxCreateDoubleMatrix(1, n, mxREAL);
            for (int i = 0; i < n; ++i) mxGetPr(a)[i] = (double)get(i);
            mxSetField(plhs[0], 0, f, a);
        };
        scalar("n_initial", ni); scalar("n_transition", info.n_transition); scalar("n_dyn", info.n_dyn);
        scalar("is_dynvar_depend", info.is_dynvar_depend);
        vec("r_initial", ni, [&](int i) { return info.r_initial[i]; });
        vec("order_initial", ni, [&](int i) { return info.order_initial[i]; });
        vec("zero_bins", ni, [&](int i) { return info.zero_bins[i]; });
        vec("resample_rates", ni, [&](int i) { return info.resample_rates[i]; });
        vec("timevarying_vars", info.n_timevarying, [&](int i) { return info.timevarying_vars[i]; });
        mxArray* tm = mxCreateDoubleMatrix(info.n_dyn, 2, mxREAL);
        for (int k = 0; k < info.n_dyn; ++k) { mxGetPr(tm)[k] = info.temporal_map[k][0]; mxGetPr(tm)[info.n_dyn + k] = info.temporal_map[k][1]; }
        mxSetField(plhs[0], 0, "temporal_map", tm);
    } else if (c == "set_prior") {                                // EncounterModel.m:194-203, setTransitionPriors.m
        CHECK(emb_set_prior(m, (int)mxGetScalar(prhs[2]), (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4])));
    } else if (c == "sample_initial") {                           // bn_sample.m:39 batch / @CorTerminalModel/sample.m
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        emb_sample_opts o;
        fill_opts(nrhs > 5 ? prhs[5] : nullptr, ni, &o);
        // MATLAB is column-major: an n x n_initial matrix IS the [n_initial][n] layout of the ABI
        plhs[0] = mxCreateNumericMatrix(n, ni, mxINT8_CLASS, mxREAL);
        mxArray* vals = mxCreateDoubleMatrix(n, ni, mxREAL);
        mxArray* att = mxCreateNumericMatrix(n, 1, mxUINT16_CLASS, mxREAL);
        CHECK(emb_sample_initial(m, &rng, n, &o, (int8_t*)mxGetData(plhs[0]), mxGetPr(vals), (uint16_t*)mxGetData(att)));
        if (nlhs > 1) plhs[1] = vals; else mxDestroyArray(vals);
        if (nlhs > 2) plhs[2] = att; else mxDestroyArray(att);
    } else if (c == "sample_tracks") {                            // UncorEncounterModel.m:244-307
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts o;
        fill_opts(nrhs > 6 ? prhs[6] : nullptr, ni, &o);
        const mwSize nch = (mwSize)((T + 3) / 4), ntile = (mwSize)((n + 127) / 128);
        // tiles [ceil(T/4)][ceil(n/128)][var][128][4] == column-major MATLAB arrays of size 4 x 128 x var x ntile x nch:
        // element (second c, track s, variable g) is A(mod(c,4)+1, mod(s,128)+1, g, floor(s/128)+1, floor(c/4)+1), 0-based c, s
        const mwSize db[5] = {4, 128, (mwSize)info.n_dyn, ntile, nch};
        const mwSize dv[5] = {4, 128, (mwSize)info.n_timevarying, ntile, nch};
        plhs[0] = mxCreateDoubleMatrix(n, ni, mxREAL);            // out_inits
        mxArray* bins = mxCreateNumericArray(5, db, mxINT8_CLASS, mxREAL);
        mxArray* vals = mxCreateNumericArray(5, dv, mxSINGLE_CLASS, mxREAL);
        mxArray* att = mxCreateNumericMatrix(n, 1, mxUINT16_CLASS, mxREAL);
        emb_track_out out{};
        out.bins = (int8_t*)mxGetData(bins);
        out.values = (float*)mxGetData(vals);
        out.init_values = mxGetPr(plhs[0]);
        out.attempts = (uint16_t*)mxGetData(att);
        CHECK(emb_sample_tracks(m, &rng, n, T, &o, &out));
        if (nlhs > 1) plhs[1] = bins; else mxDestroyArray(bins);
        if (nlhs > 2) plhs[2] = vals; else mxDestroyArray(vals);
        if (nlhs > 3) plhs[3] = att; else mxDestroyArray(att);
    } else if (c == "em_sample_text") {                           // em_sample.m:88-100: the rows of initial.txt and transition.txt
        // [initial, transition] = emb_mex('em_sample_text', h, seed, first, n, T, opts): uint8 row vectors (the files without
        // their header lines), tracks first .. first+n-1 with ids first+1 .. first+n, numbers formatted on the GPU as "%g"
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts o;
        fill_opts(nrhs > 6 ? prhs[6] : nullptr, ni, &o);
        // The MEX side has host buffers only (the ABI hands out no device memory), so the samples land in host vectors and
        // emb_format_em_sample stages them back to the device in each of its two calls: about 100 MB of extra PCIe traffic per
        // 65,536 x 60 s chunk of cor_v1.  The Python em_sample keeps them on the device and moves only the text.
        std::vector<double> inits((size_t)n * (size_t)ni);
        std::vector<float> vals((size_t)emb_tracks_values_len(m, n, T));
        emb_track_out out{};
        out.init_values = inits.data();
        out.values = vals.data();
        CHECK(emb_sample_tracks(m, &rng, n, T, &o, &out));
        std::vector<int64_t> off_i((size_t)n + 1), off_t((size_t)n + 1);
        int64_t total[2] = {0, 0};
        const int64_t first_id = (int64_t)rng.first_sample + 1;
        const int rc = emb_format_em_sample(m, n, T, first_id, inits.data(), vals.data(), &o, 0, nullptr, off_i.data(), 0, nullptr,
                                            off_t.data(), total);   // sizes both texts
        if (rc != 0 && rc != EMB_E_LIMIT) fail(rc);
        plhs[0] = mxCreateNumericMatrix(1, (mwSize)total[0], mxUINT8_CLASS, mxREAL);
        mxArray* tr = mxCreateNumericMatrix(1, (mwSize)total[1], mxUINT8_CLASS, mxREAL);
        if (rc == EMB_E_LIMIT)
            CHECK(emb_format_em_sample(m, n, T, first_id, inits.data(), vals.data(), &o, total[0], (char*)mxGetData(plhs[0]),
                                       off_i.data(), total[1], (char*)mxGetData(tr), off_t.data(), total));
        if (nlhs > 1) plhs[1] = tr; else mxDestroyArray(tr);
    } else if (c == "loglik_initial") {                           // log p of initial states (emb200.h: emb_loglik_initial)
        // [total, per_var] = emb_mex('loglik_initial', h, bins)   bins: n x n_initial int8 (== the ABI's [n_initial][n])
        const int64_t n = (int64_t)mxGetM(prhs[2]);
        if ((int64_t)mxGetNumberOfElements(prhs[2]) != n * ni) mexErrMsgIdAndTxt("emb200:arg", "bins must be an int8 n x n_initial matrix");
        emb_sample_opts o;
        emb_sample_opts_init(&o);
        plhs[0] = mxCreateDoubleMatrix(n, 1, mxREAL);
        mxArray* pv = mxCreateDoubleMatrix(n, ni, mxREAL);
        CHECK(emb_loglik_initial(m, n, (const int8_t*)mxGetData(prhs[2]), &o, mxGetPr(plhs[0]), mxGetPr(pv)));
        if (nlhs > 1) plhs[1] = pv; else mxDestroyArray(pv);
    } else if (c == "loglik_tracks") {                            // log p of tracks (emb200.h: emb_loglik_tracks)
        // [initial, transition] = emb_mex('loglik_tracks', h, init_bins, bins, T, correct_dbn)
        //   init_bins: n x n_initial int8; bins: the tiled int8 array of 'sample_tracks'
        const int64_t n = (int64_t)mxGetM(prhs[2]);
        if ((int64_t)mxGetNumberOfElements(prhs[2]) != n * ni) mexErrMsgIdAndTxt("emb200:arg", "init_bins must be an int8 n x n_initial matrix");
        const int32_t T = (int32_t)mxGetScalar(prhs[4]);
        if ((int64_t)mxGetNumberOfElements(prhs[3]) != emb_tracks_bins_len(m, n, T))
            mexErrMsgIdAndTxt("emb200:arg", "bins must be the tiled array of n tracks x T seconds");
        emb_sample_opts o;
        emb_sample_opts_init(&o);
        o.correct_dbn = nrhs > 5 ? (int32_t)mxGetScalar(prhs[5]) : 0;
        plhs[0] = mxCreateDoubleMatrix(n, 1, mxREAL);
        mxArray* tr = mxCreateDoubleMatrix(n, 1, mxREAL);
        CHECK(emb_loglik_tracks(m, n, T, (const int8_t*)mxGetData(prhs[2]), (const int8_t*)mxGetData(prhs[3]), &o,
                                mxGetPr(plhs[0]), mxGetPr(tr)));
        if (nlhs > 1) plhs[1] = tr; else mxDestroyArray(tr);
    } else if (c == "loglik_events") {                            // log p of event lists (emb200.h: emb_loglik_track_events)
        // [initial, transition] = emb_mex('loglik_events', h, init_bins, events, offsets, T, correct_dbn)
        const int64_t n = (int64_t)mxGetM(prhs[2]);
        if ((int64_t)mxGetNumberOfElements(prhs[2]) != n * ni)
            mexErrMsgIdAndTxt("emb200:arg", "init_bins must be an int8 n x n_initial matrix");
        if (mxGetM(prhs[3]) != 4)
            mexErrMsgIdAndTxt("emb200:arg", "events must be the 4 x rows [dt; var; value; bin] matrix of 'sample_events' "
                                            "(a 3-row out_events has no bins to score)");
        if ((int64_t)mxGetNumberOfElements(prhs[4]) != n + 1)
            mexErrMsgIdAndTxt("emb200:arg", "offsets must be the (n+1) x 1 offsets of 'sample_events'");
        const int64_t rows = (int64_t)mxGetNumberOfElements(prhs[3]) / 4;
        const double* e = mxGetPr(prhs[3]);
        std::vector<emb_event> ev((size_t)rows + 1);
        for (int64_t k = 0; k < rows; ++k) {
            const double dt = e[4 * k], var = e[4 * k + 1], bin = e[4 * k + 3];
            if (!(dt >= 0 && dt <= 65535 && var >= 0 && var <= 255 && bin >= 0 && bin <= 255))
                mexErrMsgIdAndTxt("emb200:arg", "events: dt, var or bin out of range in row %lld", (long long)k + 1);
            ev[(size_t)k] = emb_event{(uint16_t)dt, (uint8_t)var, (uint8_t)bin, (float)e[4 * k + 2]};
        }
        std::vector<int64_t> off((size_t)n + 1);
        for (int64_t k = 0; k <= n; ++k) off[(size_t)k] = (int64_t)mxGetPr(prhs[4])[k];
        if (off[(size_t)n] > rows) mexErrMsgIdAndTxt("emb200:arg", "offsets(end) exceeds the number of event rows");
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts o;
        emb_sample_opts_init(&o);
        o.correct_dbn = nrhs > 6 ? (int32_t)mxGetScalar(prhs[6]) : 0;
        plhs[0] = mxCreateDoubleMatrix(n, 1, mxREAL);
        mxArray* tr = mxCreateDoubleMatrix(n, 1, mxREAL);
        CHECK(emb_loglik_track_events(m, n, T, (const int8_t*)mxGetData(prhs[2]), ev.data(), off.data(), &o, mxGetPr(plhs[0]),
                                      mxGetPr(tr)));
        if (nlhs > 1) plhs[1] = tr; else mxDestroyArray(tr);
    } else if (c == "sample_tracks_multi") {                    // every GPU of the box from one MATLAB process (SURVEY 8e)
        // [out_inits, bins, values, hist_initial, hist_transition] = emb_mex('sample_tracks_multi', h, seed, first, n, T, opts, n_devices)
        // out_inits n x n_initial; bins / values: 1 x D cells of the per-device tiled arrays (shard d = emb_shard_range(n, d, D))
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts o;
        fill_opts(nrhs > 6 ? prhs[6] : nullptr, ni, &o);
        int D = nrhs > 7 ? (int)mxGetScalar(prhs[7]) : 0;
        if (D <= 0) D = emb_device_count();
        if (D <= 0) mexErrMsgIdAndTxt("emb200:cuda", "no CUDA device available");
        const mwSize nch = (mwSize)((T + 3) / 4);
        std::vector<emb_track_out> outs((size_t)D);
        std::vector<std::vector<double>> inits((size_t)D);
        mxArray* cb = mxCreateCellMatrix(1, (mwSize)D);
        mxArray* cv = mxCreateCellMatrix(1, (mwSize)D);
        for (int d = 0; d < D; ++d) {
            int64_t first = 0, cnt = 0;
            emb_shard_range(n, d, D, &first, &cnt);
            const mwSize ntile = (mwSize)((cnt + 127) / 128);
            const mwSize db[5] = {4, 128, (mwSize)info.n_dyn, ntile, nch}, dv[5] = {4, 128, (mwSize)info.n_timevarying, ntile, nch};
            mxArray* b = mxCreateNumericArray(5, db, mxINT8_CLASS, mxREAL);
            mxArray* v = mxCreateNumericArray(5, dv, mxSINGLE_CLASS, mxREAL);
            mxSetCell(cb, (mwSize)d, b);
            mxSetCell(cv, (mwSize)d, v);
            inits[(size_t)d].assign((size_t)cnt * (size_t)ni + 1, 0.0);
            outs[(size_t)d] = emb_track_out{};
            outs[(size_t)d].bins = (int8_t*)mxGetData(b);
            outs[(size_t)d].values = (float*)mxGetData(v);
            outs[(size_t)d].init_values = inits[(size_t)d].data();
        }
        mxArray* hi = mxCreateNumericMatrix(64, ni, mxUINT64_CLASS, mxREAL);          // [n_initial][64] == 64 x n_initial
        mxArray* ht = mxCreateNumericMatrix(64, info.n_dyn, mxUINT64_CLASS, mxREAL);
        const int rc = emb_sample_tracks_multi(m, &rng, n, T, &o, D, outs.data(), (unsigned long long*)mxGetData(hi),
                                               (unsigned long long*)mxGetData(ht));
        if (rc != 0) mexErrMsgIdAndTxt("emb200:error", "%s", emb_multi_last_error());
        plhs[0] = mxCreateDoubleMatrix(n, ni, mxREAL);                                // shards back to back: out_inits
        for (int d = 0; d < D; ++d) {
            int64_t first = 0, cnt = 0;
            emb_shard_range(n, d, D, &first, &cnt);
            for (int i = 0; i < ni; ++i)
                std::memcpy(mxGetPr(plhs[0]) + (size_t)i * (size_t)n + (size_t)first, inits[(size_t)d].data() + (size_t)i * (size_t)cnt,
                            (size_t)cnt * 8);
        }
        if (nlhs > 1) plhs[1] = cb; else mxDestroyArray(cb);
        if (nlhs > 2) plhs[2] = cv; else mxDestroyArray(cv);
        if (nlhs > 3) plhs[3] = hi; else mxDestroyArray(hi);
        if (nlhs > 4) plhs[4] = ht; else mxDestroyArray(ht);
    } else if (c == "tracks_integrate") {                         // sample2track.m:188-244
        const int64_t n = (int64_t)mxGetM(prhs[2]);
        const int32_t T = (int32_t)mxGetScalar(prhs[4]);
        const mxArray* io = prhs[5];
        emb_integrate_opts o;
        std::memset(&o, 0, sizeof(o));
        o.idx_altitude = (int)field_or(io, "idx_altitude", 0); o.idx_speed = (int)field_or(io, "idx_speed", 0);
        o.idx_acceleration = (int)field_or(io, "idx_acceleration", 0); o.idx_vertrate = (int)field_or(io, "idx_vertrate", 0);
        o.idx_turnrate = (int)field_or(io, "idx_turnrate", 0);
        o.ur_speed = field_or(io, "ur_speed", 6076.1154855643 / 3600); o.ur_vertrate = field_or(io, "ur_vertrate", 1.0 / 60);
        o.ur_heading = field_or(io, "ur_heading", 1.0);
        o.min_speed = field_or(io, "min_speed", 0); o.max_speed = field_or(io, "max_speed", 1e300);
        o.mem = EMB_MEM_HOST; o.device = -1;
        const mwSize dx[3] = {(mwSize)n, (mwSize)(T + 1), 3};      // [3][T+1][n] == n x (T+1) x 3 column-major
        plhs[0] = mxCreateNumericArray(3, dx, mxSINGLE_CLASS, mxREAL);
        mxArray* good = mxCreateNumericMatrix(n, 1, mxUINT8_CLASS, mxREAL);
        CHECK(emb_tracks_integrate(m, n, T, mxGetPr(prhs[2]), (const float*)mxGetData(prhs[3]), &o, (float*)mxGetData(plhs[0]),
                                   (uint8_t*)mxGetData(good)));
        if (nlhs > 1) plhs[1] = good; else mxDestroyArray(good);
    } else if (c == "sample_tracks_xyz") {                        // sample2track.m:150-244 in one pass
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts so;
        fill_opts(nrhs > 6 ? prhs[6] : nullptr, ni, &so);
        const mxArray* io = nrhs > 7 ? prhs[7] : nullptr;
        emb_integrate_opts o;
        std::memset(&o, 0, sizeof(o));
        o.idx_altitude = (int)field_or(io, "idx_altitude", 0); o.idx_speed = (int)field_or(io, "idx_speed", 0);
        o.idx_acceleration = (int)field_or(io, "idx_acceleration", 0); o.idx_vertrate = (int)field_or(io, "idx_vertrate", 0);
        o.idx_turnrate = (int)field_or(io, "idx_turnrate", 0);
        o.ur_speed = field_or(io, "ur_speed", 6076.1154855643 / 3600); o.ur_vertrate = field_or(io, "ur_vertrate", 1.0 / 60);
        o.ur_heading = field_or(io, "ur_heading", 1.0);
        o.min_speed = field_or(io, "min_speed", 0); o.max_speed = field_or(io, "max_speed", 1e300);
        const mwSize dx[3] = {(mwSize)n, (mwSize)(T + 1), 3};      // [3][T+1][n] == n x (T+1) x 3 column-major
        plhs[0] = mxCreateNumericArray(3, dx, mxSINGLE_CLASS, mxREAL);
        mxArray* good = mxCreateNumericMatrix(n, 1, mxUINT8_CLASS, mxREAL);
        mxArray* inits = mxCreateDoubleMatrix(n, ni, mxREAL);
        emb_track_out out{};
        out.init_values = mxGetPr(inits);
        CHECK(emb_sample_tracks_xyz(m, &rng, n, T, &so, &o, &out, (float*)mxGetData(plhs[0]), (uint8_t*)mxGetData(good)));
        if (nlhs > 1) plhs[1] = good; else mxDestroyArray(good);
        if (nlhs > 2) plhs[2] = inits; else mxDestroyArray(inits);
    } else if (c == "sample_events") {                            // out_events of UncorEncounterModel.m:253-300
        emb_rng rng{(uint64_t)mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])};
        const int64_t n = (int64_t)mxGetScalar(prhs[4]);
        const int32_t T = (int32_t)mxGetScalar(prhs[5]);
        emb_sample_opts o;
        fill_opts(nrhs > 6 ? prhs[6] : nullptr, ni, &o);
        std::vector<int64_t> off((size_t)n + 1);
        mxArray* inits = mxCreateDoubleMatrix(n, ni, mxREAL);
        mxArray* att = mxCreateNumericMatrix(n, 1, mxUINT16_CLASS, mxREAL);
        mxArray* ibins = mxCreateNumericMatrix(n, ni, mxINT8_CLASS, mxREAL);   // n x n_initial == the ABI's [n_initial][n]
        emb_track_out init{};
        init.init_values = mxGetPr(inits);
        init.attempts = (uint16_t*)mxGetData(att);
        init.init_bins = (int8_t*)mxGetData(ibins);
        int64_t total = 0;
        std::vector<uint32_t> words;
        std::vector<uint8_t> dts;
        std::vector<emb_event> ev;
        // 5-byte packed rows (what the device writes and what crosses PCIe); the value of a row is evaluated here in fp64 from
        // its bin and 23-bit uniform exactly as dediscretize.m:39 does.  Models outside the packed format (more than 7
        // time-varying variables or T > 1023) take the 8-byte rows.
        int rc = emb_sample_track_events_packed(m, &rng, n, T, &o, 0, nullptr, nullptr, off.data(), &init, &total);   // sizes the list
        const bool packed = rc == 0 || (rc == EMB_E_LIMIT && total > 0);
        if (packed) {
            words.resize((size_t)total + 1);
            dts.resize((size_t)total + 1);
            CHECK(emb_sample_track_events_packed(m, &rng, n, T, &o, total, words.data(), dts.data(), off.data(), &init, &total));
            int32_t gated[EMB_MAX_GATED];
            const int ng = (int)emb_model_get_gated(m, gated, EMB_MAX_GATED);
            std::vector<double> bnd((size_t)emb_model_get_boundaries(m, nullptr, 0) + 1);
            emb_model_get_boundaries(m, bnd.data(), (int64_t)bnd.size());
            std::vector<int64_t> boff((size_t)ni + 1, 0);
            for (int i = 0; i < ni; ++i) boff[(size_t)i + 1] = boff[(size_t)i] + info.boundaries_len[i];
            plhs[0] = mxCreateDoubleMatrix(4, (mwSize)total, mxREAL);
            double* e = mxGetPr(plhs[0]);
            for (int64_t k = 0; k < total; ++k) {
                const uint32_t w = words[(size_t)k], gord = (w >> 27) & 7u;
                const double dt = (double)(dts[(size_t)k] | ((w >> 30) << 8));
                double var = 0, val = 0, bin = 0;
                if (gord > 0 && (int)gord <= ng) {
                    const int v = gated[gord - 1];                       // 1-based variable id
                    const int b = (int)((w >> 23) & 15u) + 1;
                    var = v; bin = b;
                    if (info.boundaries_len[v - 1] == 0) val = b;                                   // dediscretize.m:7-10
                    else if (info.zero_bins[v - 1] == b) val = 0.0;                                 // :24-25
                    else {
                        const double* ed = bnd.data() + boff[(size_t)v - 1];
                        const double u = ((double)(w & 0x7FFFFFu) + 0.5) * 1.1920928955078125e-07;  // (frac + 0.5) 2^-23
                        val = ed[b - 1] + (ed[b] - ed[b - 1]) * u;                                  // :39
                    }
                }
                e[4 * k] = dt; e[4 * k + 1] = var; e[4 * k + 2] = val; e[4 * k + 3] = bin;
            }
        } else {
        rc = emb_sample_track_events(m, &rng, n, T, &o, 0, nullptr, off.data(), &init, &total);   // sizes the list
        if (rc != 0 && rc != EMB_E_LIMIT) fail(rc);
        ev.resize((size_t)total + 1);
        CHECK(emb_sample_track_events(m, &rng, n, T, &o, total, ev.data(), off.data(), &init, &total));
        plhs[0] = mxCreateDoubleMatrix(4, (mwSize)total, mxREAL);
        double* e = mxGetPr(plhs[0]);
        for (int64_t k = 0; k < total; ++k) {
            e[4 * k] = ev[(size_t)k].dt; e[4 * k + 1] = ev[(size_t)k].var; e[4 * k + 2] = ev[(size_t)k].value; e[4 * k + 3] = ev[(size_t)k].bin;
        }
        }
        mxArray* offs = mxCreateDoubleMatrix(n + 1, 1, mxREAL);
        for (int64_t k = 0; k <= n; ++k) mxGetPr(offs)[k] = (double)off[(size_t)k];
        if (nlhs > 1) plhs[1] = offs; else mxDestroyArray(offs);
        if (nlhs > 2) plhs[2] = inits; else mxDestroyArray(inits);
        if (nlhs > 3) plhs[3] = att; else mxDestroyArray(att);
        if (nlhs > 4) plhs[4] = ibins; else mxDestroyArray(ibins);
        if (nlhs > 5) {   // out_samples and the out_EME matrices on the GPU, from the rows above (host buffers)
            emb_controls_spec spec{};
            if (nlhs > 6) {   // UncorEncounterModel.m:225-234, 286-297
                std::string lab((size_t)emb_model_get_labels(m, 0, nullptr, 0), '\0');
                emb_model_get_labels(m, 0, &lab[0], (int64_t)lab.size());
                auto find = [&](const char* name) {
                    int id = 1;
                    for (size_t a = 0; a < lab.size();) {
                        const size_t b = std::min(lab.find('\n', a), lab.size() - 1);
                        if (lab.compare(a, b - a, name) == 0) return id;
                        a = b + 1;
                        ++id;
                    }
                    mexErrMsgIdAndTxt("dynvar:empty", "Model does not have a dynamic variable for either acceleration, vertical "
                                                      "rate, or turn rate");
                    return 0;
                };
                spec.n_cols = 3;
                spec.vars[0] = find("\"\\dot h\"");
                spec.vars[1] = find("\"\\dot \\psi\"");
                spec.vars[2] = find("\"\\dot v\"");
                const double mul[3] = {1.0, 3.141592653589793 / 180.0, 1.68780972222222}, div[3] = {60.0, 1.0, 1.0};
                for (int j = 0; j < 3; ++j) {
                    spec.mul[j] = mul[j];
                    spec.div[j] = div[j];
                }
            }
            emb_sample_opts eo;
            emb_sample_opts_init(&eo);
            eo.device = o.device;
            std::vector<double> smp((size_t)n * (size_t)T * (size_t)ni);
            std::vector<int64_t> coff((size_t)n + 1);
            std::vector<double> rows;
            int64_t ctl_total = 0;
            auto expand = [&](int64_t capacity, double* r, int64_t* co, int64_t* tot) {
                return packed ? emb_track_events_expand_packed(m, n, T, mxGetPr(inits), words.data(), dts.data(), off.data(), &eo,
                                                               &spec, smp.data(), capacity, r, co, tot)
                              : emb_track_events_expand(m, n, T, mxGetPr(inits), ev.data(), off.data(), &eo, &spec, smp.data(),
                                                        capacity, r, co, tot);
            };
            if (nlhs > 6) {
                rc = expand(0, nullptr, coff.data(), &ctl_total);   // sizes the control rows
                if (rc != 0 && rc != EMB_E_LIMIT) fail(rc);
                rows.resize((size_t)ctl_total * 4 + 1);
                CHECK(expand(ctl_total, rows.data(), coff.data(), &ctl_total));
            } else {
                CHECK(expand(0, nullptr, nullptr, nullptr));
            }
            plhs[5] = mxCreateCellMatrix(n, 1);
            for (int64_t s = 0; s < n; ++s) {
                mxArray* x = mxCreateDoubleMatrix(ni, T, mxREAL);   // [T][n_initial] of track s is the column-major ni x T
                std::memcpy(mxGetPr(x), smp.data() + (size_t)s * T * ni, sizeof(double) * (size_t)T * ni);
                mxSetCell(plhs[5], s, x);
            }
            if (nlhs > 6) {
                plhs[6] = mxCreateCellMatrix(n, 1);
                for (int64_t s = 0; s < n; ++s) {
                    const int64_t k = coff[(size_t)s + 1] - coff[(size_t)s];
                    mxArray* x = mxCreateDoubleMatrix(k, 4, mxREAL);
                    double* pr = mxGetPr(x);
                    const double* r = rows.data() + (size_t)coff[(size_t)s] * 4;
                    for (int64_t q = 0; q < k; ++q)
                        for (int c = 0; c < 4; ++c) pr[c * k + q] = r[q * 4 + c];
                    mxSetCell(plhs[6], s, x);
                }
            }
        }
    } else {
        mexErrMsgIdAndTxt("emb200:arg", "unknown command '%s'", cmd);
    }
}
