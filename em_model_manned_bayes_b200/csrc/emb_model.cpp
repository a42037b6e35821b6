// emb_model.cpp -- model reader and packer (host only, no CUDA).
//
// Reader semantics follow /root/reference/code/matlab/em_read.m:47-141 (+ helpers :143-206) and
// bn_sort.m:14-24; nothing is shared with oracle/ (the oracle has its own restatement, and the two
// are compared in tests/test_reader.py).  The packer is new: it converts each column of
// N + alpha into the word-space threshold form documented in emb_device.cuh.
#include "emb_model.h"

#include <algorithm>
#include <cctype>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <limits>
#include <memory>
#include <queue>
#include <sstream>

#include "../../include/emb200.h"

namespace emb {

namespace {

[[noreturn]] void fail(int code, const std::string& msg) { throw Error{code, msg}; }

std::string trim(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && (s[a] == ' ' || s[a] == '\t')) ++a;
    while (b > a && (s[b - 1] == ' ' || s[b - 1] == '\t')) --b;
    return s.substr(a, b - a);
}

// textscan(line, '%f', 'Delimiter', ' ') : numbers until the first token that is not a number
void scan_numbers(const std::string& line, std::vector<double>& out) {
    const char* p = line.c_str();
    const char* end = p + line.size();
    while (p < end) {
        while (p < end && (*p == ' ' || *p == '\t' || *p == ',')) ++p;
        if (p >= end) break;
        char* q = nullptr;
        errno = 0;
        const double v = std::strtod(p, &q);
        if (q == p) break;
        out.push_back(v);
        p = q;
    }
}

std::vector<std::string> split_labels(const std::string& line) {
    std::vector<std::string> out;
    std::string cur;
    std::stringstream ss(line);
    while (std::getline(ss, cur, ',')) out.push_back(trim(cur));  // strtrim(strsplit(line, ','))
    return out;
}

// bn_sort.m:14-24 -> toposort(digraph(G),'Order','stable'): smallest ready index first
std::vector<int32_t> topo_sort(const std::vector<uint8_t>& G, int n) {
    std::vector<int> indeg(n, 0);
    for (int p = 0; p < n; ++p)
        for (int c = 0; c < n; ++c) indeg[c] += G[(size_t)p * n + c] ? 1 : 0;
    std::priority_queue<int, std::vector<int>, std::greater<int>> ready;
    for (int i = 0; i < n; ++i)
        if (!indeg[i]) ready.push(i);
    std::vector<int32_t> order;
    while (!ready.empty()) {
        const int i = ready.top();
        ready.pop();
        order.push_back(i);
        for (int c = 0; c < n; ++c)
            if (G[(size_t)i * n + c] && --indeg[c] == 0) ready.push(c);
    }
    if ((int)order.size() != n) fail(EMB_E_MODEL, "Network could not be hierarchically sorted");
    return order;
}

void parse_matrix(const std::vector<std::string>& lines, size_t row, int n, std::vector<uint8_t>& G, const char* what) {
    G.assign((size_t)n * n, 0);
    for (int i = 0; i < n; ++i) {
        if (row + i >= lines.size()) fail(EMB_E_PARSE, std::string("truncated field ") + what);
        std::vector<double> v;
        scan_numbers(lines[row + i], v);
        if ((int)v.size() != n) fail(EMB_E_PARSE, std::string("bad row length in ") + what);
        for (int c = 0; c < n; ++c) G[(size_t)i * n + c] = v[c] != 0.0;
    }
}

// em_read.m:200-206 getdims + :191-198 array2cells
void fill_tables(const std::vector<uint8_t>& G, const std::vector<int32_t>& r, int n, int first, int last,
                 const std::vector<double>& x, std::vector<Table>& T, const char* what) {
    T.assign(n, Table{});
    size_t index = 0;
    for (int i = first; i < last; ++i) {
        Table& t = T[i];
        t.r = r[i];
        t.q = 1;
        for (int p = 0; p < n; ++p)
            if (G[(size_t)p * n + i]) {
                t.parents.push_back(p);
                t.q *= r[p];
            }
        const size_t cnt = (size_t)t.r * (size_t)t.q;
        if (index + cnt > x.size()) fail(EMB_E_PARSE, std::string(what) + " is shorter than sum(r_i*q_i)");
        t.N.assign(x.begin() + index, x.begin() + index + cnt);
        t.present = true;
        index += cnt;
    }
    if (index != x.size()) fail(EMB_E_PARSE, std::string(what) + " is longer than sum(r_i*q_i)");
}

}  // namespace

// ------------------------------------------------------------------------------------------------
uint64_t gate_threshold(double rate) {
    if (!(rate > 0.0)) return 0;
    if (rate >= 1.0) return 1ull << 32;
    auto fires = [rate](uint64_t k) { return ((double)k + 0.5) * 2.3283064365386963e-10 < rate; };
    uint64_t g = (uint64_t)std::floor(rate * 4294967296.0);
    if (g > 0xFFFFFFFFull) g = 0xFFFFFFFFull;
    while (g > 0 && !fires(g - 1)) --g;
    while (g < (1ull << 32) && fires(g)) ++g;
    return g;
}

void pack_column(const double* w, int r, int rp, uint32_t* col) {
    // s = cumsum(w) sequentially in fp64 (select_random.m:17)
    double s[256];
    double acc = 0.0;
    for (int m = 0; m < r; ++m) {
        acc += w[m];
        s[m] = acc;
    }
    const double total = s[r - 1];
    for (int m = 0; m < rp; ++m) col[m] = 0xFFFFFFFFu;
    uint32_t lead = 0;
    uint64_t lo_bound = 0;
    for (int m = 0; m + 1 < r; ++m) {
        // K_m = min{k in [0, 2^32] : s[m] < fl(total * u_k)};  predicate is monotone in k
        const double sm = s[m];
        auto above = [total, sm](uint64_t k) {
            const double u = ((double)k + 0.5) * 2.3283064365386963e-10;   // exact
            volatile double thr = total * u;                                // select_random.m:18
            return !(sm >= thr);                                            // :19 x = s >= sthres
        };
        uint64_t lo = lo_bound, hi = 1ull << 32;  // answer in [lo, hi]
        if (!(total > 0.0) || std::isnan(total)) {
            lo = hi;  // all-zero (or NaN) column: s >= 0 always holds -> bin 1
        } else {
            while (lo < hi) {
                const uint64_t mid = lo + ((hi - lo) >> 1);
                if (above(mid)) hi = mid; else lo = mid + 1;
            }
        }
        lo_bound = lo;
        if (lo == 0) ++lead;
        else col[m] = (uint32_t)(lo - 1);  // lo == 2^32 -> 0xFFFFFFFF (never)
    }
    col[rp - 1] = lead;
}

void logp_column(const double* w, int r, int rp, double* col) {
    double total = 0.0;
    for (int m = 0; m < r; ++m) total += w[m];
    const double ninf = -std::numeric_limits<double>::infinity();
    for (int m = 0; m < rp; ++m) col[m] = ninf;
    if (!(total > 0.0)) {
        col[0] = 0.0;
        return;
    }
    for (int m = 0; m < r; ++m)
        if (w[m] > 0.0) col[m] = std::log(w[m] / total);
}

// ------------------------------------------------------------------------------------------------
HostModel* load_model_file(const char* path, bool overwrite_zero_boundaries, const int32_t* idx_zero, int n_idx) {
    std::ifstream f(path, std::ios::binary);
    if (!f) fail(EMB_E_IO, std::string("cannot open parameters file: ") + path);
    std::string raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    // textscan(fid,'%s','EndOfLine','\r\n','Whitespace','\r\n') : split on CR / LF, drop blank lines
    std::vector<std::string> lines;
    {
        std::string cur;
        for (char ch : raw) {
            if (ch == '\r' || ch == '\n') {
                if (!trim(cur).empty()) lines.push_back(cur);
                cur.clear();
            } else {
                cur.push_back(ch);
            }
        }
        if (!trim(cur).empty()) lines.push_back(cur);
    }
    std::unique_ptr<HostModel> M(new HostModel());
    std::vector<double> xs;
    for (size_t li = 0; li < lines.size(); ++li) {
        if (lines[li].find('#') == std::string::npos) continue;  // em_read.m:54
        const std::string name = trim(lines[li]);
        const size_t row = li + 1;
        auto need = [&](size_t k) {
            if (row + k > lines.size()) fail(EMB_E_PARSE, "truncated field " + name);
        };
        if (name == "# labels_initial") {
            need(1);
            M->labels_initial = split_labels(lines[row]);
            M->n_initial = (int32_t)M->labels_initial.size();
        } else if (name == "# G_initial") {
            parse_matrix(lines, row, M->n_initial, M->G_initial, "G_initial");
            M->order_initial = topo_sort(M->G_initial, M->n_initial);  // em_read.m:74: bn_sort at parse time
        } else if (name == "# r_initial") {
            need(1);
            xs.clear();
            scan_numbers(lines[row], xs);
            M->r_initial.assign(xs.begin(), xs.end());
        } else if (name == "# N_initial") {
            need(1);
            if ((int)M->r_initial.size() != M->n_initial || M->G_initial.empty())
                fail(EMB_E_PARSE, "N_initial before G_initial/r_initial");
            xs.clear();
            scan_numbers(lines[row], xs);
            fill_tables(M->G_initial, M->r_initial, M->n_initial, 0, M->n_initial, xs, M->T_initial, "N_initial");
        } else if (name == "# labels_transition") {
            need(1);
            M->labels_transition = split_labels(lines[row]);
            M->n_transition = (int32_t)M->labels_transition.size();
            M->has_transition = true;
        } else if (name == "# G_transition") {
            parse_matrix(lines, row, M->n_transition, M->G_transition, "G_transition");
            M->order_transition = topo_sort(M->G_transition, M->n_transition);  // em_read.m:87
        } else if (name == "# r_transition") {
            need(1);
            xs.clear();
            scan_numbers(lines[row], xs);
            M->r_transition.assign(xs.begin(), xs.end());
        } else if (name == "# N_transition") {
            need(1);
            if ((int)M->r_transition.size() != M->n_transition || M->G_transition.empty())
                fail(EMB_E_PARSE, "N_transition before G_transition/r_transition");
            xs.clear();
            scan_numbers(lines[row], xs);
            fill_tables(M->G_transition, M->r_transition, M->n_transition, M->n_initial, M->n_transition, xs,
                        M->T_transition, "N_transition");  // em_read.m:92
        } else if (name == "# boundaries") {
            need((size_t)M->n_initial);
            M->boundaries.assign(M->n_initial, {});
            for (int j = 0; j < M->n_initial; ++j) scan_numbers(lines[row + j], M->boundaries[j]);
            M->has_boundaries = true;
        } else if (name == "# resample_rates") {
            need(1);
            xs.clear();
            scan_numbers(lines[row], xs);
            M->resample_rates = xs;
        } else {
            fail(EMB_E_PARSE, "Unknown field: " + name);  // em_read.m:105
        }
    }
    if (M->n_initial <= 0 || M->T_initial.empty()) fail(EMB_E_PARSE, "missing labels_initial / N_initial");
    M->derive();
    if (overwrite_zero_boundaries && M->has_boundaries) {  // em_read.m:119-121 (after zero-bin extraction)
        for (int k = 0; k < n_idx; ++k) {
            const int v = idx_zero[k] - 1;
            if (v >= 0 && v < M->n_initial) M->boundaries[v].clear();
        }
        // bounds_initial of an emptied variable is [0 0] (em_read.m:129-131)
        for (int i = 0; i < M->n_initial; ++i)
            if (M->boundaries[i].empty()) M->bounds_initial[i] = {0.0, 0.0};
    }
    M->pack();
    return M.release();
}

// ------------------------------------------------------------------------------------------------
void HostModel::derive() {
    const int n = n_initial;
    if (n > MAXV) fail(EMB_E_LIMIT, "model has more than EMB_MAX_VARS initial variables");
    if ((int)r_initial.size() != n) fail(EMB_E_PARSE, "r_initial length mismatch");
    for (int i = 0; i < n; ++i)
        if (r_initial[i] < 1 || r_initial[i] > 127) fail(EMB_E_LIMIT, "r_initial out of range [1,127]");
    order_initial = topo_sort(G_initial, n);
    if (boundaries.empty()) boundaries.assign(n, {});
    if (resample_rates.empty()) resample_rates.assign(n, 0.0);
    if ((int)resample_rates.size() != n) fail(EMB_E_PARSE, "resample_rates length mismatch");
    // zero bins (em_read.m:143-156) and bounds (em_read.m:124-136)
    zero_bins.assign(n, 0);
    bounds_initial.assign(n, {0.0, 0.0});
    for (int i = 0; i < n; ++i) {
        const auto& b = boundaries[i];
        if (!b.empty() && (int)b.size() != r_initial[i] + 1)
            fail(EMB_E_PARSE, "boundaries of variable " + std::to_string(i + 1) + " must have r+1 edges");
        if (b.size() > 2)
            for (size_t j = 1; j < b.size(); ++j)
                if (b[j - 1] < 0 && b[j] > 0) zero_bins[i] = (int32_t)j;
        if (!b.empty()) bounds_initial[i] = {*std::min_element(b.begin(), b.end()), *std::max_element(b.begin(), b.end())};
    }
    if (!temporal_map_given) temporal_map.clear();
    is_dynvar_depend = false;
    if (has_transition) {
        if (n_transition > MAXX) fail(EMB_E_LIMIT, "too many transition variables");
        if ((int)r_transition.size() != n_transition) fail(EMB_E_PARSE, "r_transition length mismatch");
        order_transition = topo_sort(G_transition, n_transition);
        // em_read.m:158-177
        for (int i = 0; i < n_transition && !temporal_map_given; ++i) {
            const std::string& lab = labels_transition[i];
            const size_t t = lab.find("(t)");
            if (t == std::string::npos) continue;
            const std::string stem = lab.substr(0, t + 1);
            for (const char* suffix : {"t+1)", "t-1)"})
                for (int k = 0; k < n_transition; ++k)
                    if (labels_transition[k].find(stem + suffix) != std::string::npos) temporal_map.push_back({i, k});
        }
        if ((int)temporal_map.size() > MAXD) fail(EMB_E_LIMIT, "more than EMB_MAX_DYN dynamic variables");
        for (auto& a : temporal_map) {
            if (a.first >= n) fail(EMB_E_MODEL, "temporal_map: variable at time t is not an initial variable");
            if (!T_transition[a.second].present) fail(EMB_E_MODEL, "dynamic variable without N_transition table");
            if (r_transition[a.second] != r_initial[a.first]) fail(EMB_E_MODEL, "r of X(t+1) differs from r of X(t)");
            for (auto& b : temporal_map)
                if (G_transition[(size_t)a.second * n_transition + b.second]) is_dynvar_depend = true;  // dbn_sample.m:55
        }
        for (int i = 0; i < n; ++i)
            if (r_transition[i] != r_initial[i]) fail(EMB_E_MODEL, "r_transition(1:n_initial) differs from r_initial");
    }
    // stream spec v5: a variable owns one word per second iff its value can change (rate > 0 or dynamic)
    gated.clear();
    for (int i = 0; i < n; ++i) {
        bool g = resample_rates[i] > 0.0;
        for (auto& a : temporal_map) g = g || a.first == i;
        if (g) gated.push_back(i);
    }
    if ((int)gated.size() > MAXG) fail(EMB_E_LIMIT, "more than EMB_MAX_GATED resampled or dynamic variables");
    timevarying.clear();
    for (int i = 0; i < n; ++i) {
        bool tv = resample_rates[i] > 0.0;
        for (auto& a : temporal_map) tv = tv || a.first == i;
        if (tv) timevarying.push_back(i);
    }
}

// ------------------------------------------------------------------------------------------------
namespace {

// weights of column j of a table under a prior
struct AlphaFn {
    int kind;
    double value;
    int r;
    int64_t q;
    int64_t stay_block;  // q / r for EMB_PRIOR_STAY
    double operator()(int m, int64_t j) const {
        switch (kind) {
            case EMB_PRIOR_DBE: return 1.0 / ((double)r * (double)q);          // bn_dirichlet_prior.m:24
            case EMB_PRIOR_STAY: return (j / stay_block) == m ? value : 0.0;   // setTransitionPriors.m:25-27
            default: return value;                                             // bn_dirichlet_prior.m:34
        }
    }
};

void pack_table(const Table& t, const PriorSpec& pr, bool stay_ok, Node& node, std::vector<uint32_t>& out,
                std::vector<double>& logp, const std::vector<int32_t>& xindex_of_parent) {
    if (t.r > 127) fail(EMB_E_LIMIT, "more than 127 bins");
    if ((int)t.parents.size() > MAXP) fail(EMB_E_LIMIT, "more than EMB_MAX_PARENTS parents");
    node.r = t.r;
    node.rp = (t.r + 3) & ~3;
    node.np = (int32_t)t.parents.size();
    node.off = (uint32_t)out.size();
    if (out.size() + (size_t)t.q * node.rp > 0xFFFFFFF0ull) fail(EMB_E_LIMIT, "threshold table exceeds 2^32 entries");
    (void)xindex_of_parent;
    AlphaFn a{pr.kind, pr.value, t.r, t.q, 1};
    if (pr.kind == EMB_PRIOR_STAY) {
        if (!stay_ok || t.q % t.r) fail(EMB_E_ARG, "stay prior needs a parent table whose column count is a multiple of r");
        a.stay_block = t.q / t.r;
    }
    out.resize(out.size() + (size_t)t.q * node.rp);
    logp.resize(out.size());
    std::vector<double> w(t.r);
    for (int64_t j = 0; j < t.q; ++j) {
        for (int m = 0; m < t.r; ++m) {
            const double v = t.N[(size_t)j * t.r + m] + a(m, j);
            if (!(v >= 0.0)) fail(EMB_E_MODEL, "negative or NaN weight in count table");
            w[m] = v;
        }
        pack_column(w.data(), t.r, node.rp, out.data() + node.off + (size_t)j * node.rp);
        logp_column(w.data(), t.r, node.rp, logp.data() + node.off + (size_t)j * node.rp);
    }
}

}  // namespace

void HostModel::pack() {
    DevModel& D = dev;
    std::memset(&D, 0, sizeof(D));
    const int n = n_initial;
    D.n_initial = n;
    D.n_transition = has_transition ? n_transition : n;
    D.n_dyn = (int32_t)temporal_map.size();
    D.n_gated = (int32_t)gated.size();
    D.n_tv = (int32_t)timevarying.size();
    D.nw = D.n_gated;   // stream spec v5: one word per (second, gated variable)
    D.fast = is_dynvar_depend ? 0 : 1;
    D.two23 = 1 << 23;
    for (int i = 0; i < n; ++i) D.order_initial[i] = order_initial[i];

    thr_initial.clear();
    thr_transition.clear();
    logp_initial.clear();
    logp_transition.clear();
    std::vector<int32_t> ident;
    for (int i = 0; i < n; ++i) {
        const Table& t = T_initial[i];
        Node& nd = D.init[i];
        pack_table(t, prior_initial, false, nd, thr_initial, logp_initial, ident);
        uint32_t stride = 1;
        for (int p = 0; p < nd.np; ++p) {  // asub2ind.m:13 strides over parents in increasing index
            nd.par[p] = (uint8_t)t.parents[p];
            nd.stride_rp[p] = stride * (uint32_t)nd.rp;
            stride *= (uint32_t)r_initial[t.parents[p]];
        }
    }
    for (int d = 0; d < D.n_dyn; ++d) {
        const int vt = temporal_map[d].first, vt1 = temporal_map[d].second;
        D.dyn_t[d] = vt;
        D.dyn_t1[d] = vt1;
        const Table& t = T_transition[vt1];
        Node& nd = D.dyn[d];
        pack_table(t, prior_transition, true, nd, thr_transition, logp_transition, ident);
        uint32_t stride = 1;
        for (int p = 0; p < nd.np; ++p) {
            nd.par[p] = (uint8_t)t.parents[p];
            nd.stride_rp[p] = stride * (uint32_t)nd.rp;
            stride *= (uint32_t)r_transition[t.parents[p]];
        }
    }
    // dynamic ordinals in order_transition order (dbn_sample.m:69)
    {
        int k = 0;
        for (int32_t v : order_transition)
            for (int d = 0; d < D.n_dyn; ++d)
                if (temporal_map[d].second == v) D.order_dyn[k++] = d;
    }
    for (int g = 0; g < D.n_gated; ++g) {
        D.gated_var[g] = gated[g];
        D.gate_G[g] = gate_threshold(resample_rates[gated[g]]);
    }
    for (int d = 0; d < D.n_dyn; ++d)
        for (int g = 0; g < D.n_gated; ++g)
            if (gated[g] == temporal_map[d].first) D.gate_of_dyn[d] = g;
    for (int i = 0; i < MAXV; ++i) D.tv_of_var[i] = -1;
    for (int k = 0; k < D.n_tv; ++k) {
        D.tv_var[k] = timevarying[k];
        D.tv_of_var[timevarying[k]] = k;
    }
    edges.clear();
    for (int i = 0; i < n; ++i) {
        D.zero_bin[i] = zero_bins[i];
        if (boundaries[i].empty()) {
            D.edge_off[i] = -1;
            continue;
        }
        D.edge_off[i] = (int32_t)edges.size();
        for (int b = 0; b < r_initial[i]; ++b) {
            const double a = boundaries[i][b];
            volatile double w = boundaries[i][b + 1] - a;  // dediscretize.m:39 (b - a)
            edges.push_back(a);
            edges.push_back((double)w);
        }
    }
    // fp32 de-discretisation entries of the gated variables, {slope, base, s, c} per bin:
    //   f in [1,2) carries the 23-bit value-word fraction g = f - 1;  g' = fma(f, s, c);  value = fma(slope, g', base)
    //   bins on the positive side: (s, c) = (1, -1), g' = g,            value = (a + w 2^-24) + w g
    //   bins on the negative side: (s, c) = (-1, 2 - 2^-23), g' = 1 - 2^-23 - g, value = (b - w 2^-24) - w g'
    // so that every term has the sign of the result and fp32 rounding stays <= ~2e-7 relative.
    dd32.clear();
    D.fast32_ok = 1;
    D.init32_ok = 1;
    auto entries_of = [&](int v, int32_t& ok) {
        for (int b = 0; b < r_initial[v]; ++b) {
            float e[4] = {0.0f, 0.0f, 1.0f, -1.0f};
            if (boundaries[v].empty()) {
                e[1] = (float)(b + 1);                                  // dediscretize.m:7-10: the bin itself
            } else if (zero_bins[v] == b + 1) {
                e[1] = 0.0f;                                            // :24-25
            } else {
                const double a = boundaries[v][b], bb = boundaries[v][b + 1];
                volatile double w = bb - a;
                if (a < 0.0 && bb > 0.0) ok = 0;                        // value can cancel to ~0: fp64 only
                if (a + bb < 0.0) {
                    e[0] = (float)(-(double)w);
                    e[1] = (float)(bb - (double)w * 5.9604644775390625e-08);
                    e[2] = -1.0f;
                    e[3] = 1.99999988079071044921875f;                  // 2 - 2^-23
                } else {
                    e[0] = (float)(double)w;
                    e[1] = (float)(a + (double)w * 5.9604644775390625e-08);
                }
            }
            dd32.insert(dd32.end(), e, e + 4);
        }
    };
    for (int g = 0; g < D.n_gated; ++g) {
        D.dd_off[g] = (int32_t)(dd32.size() / 4);
        entries_of(gated[g], D.fast32_ok);
    }
    for (int i = 0; i < n_initial; ++i) {                               // all initial variables (emb_initial.cuh, fp32 values)
        D.ddi_off[i] = (int32_t)(dd32.size() / 4);
        entries_of(i, D.init32_ok);
    }
    ++version;
}

// Validate caller options against the model and translate them into the kernel parameter block.
void fill_params(const HostModel& H, uint64_t seed, uint64_t first_sample, int64_t n, int32_t T,
                 const emb_sample_opts& opts, SampleParams& P) {
    const emb_sample_opts* o = &opts;
    std::memset(&P, 0, sizeof(P));
    P.seed = seed;
    for (int i = 0; i < 10; ++i) {
        P.rk[2 * i] = (uint32_t)seed + (uint32_t)i * PHILOX_W0;
        P.rk[2 * i + 1] = (uint32_t)(seed >> 32) + (uint32_t)i * PHILOX_W1;
    }
    P.first_sample = first_sample;
    P.n = n;
    P.s_begin = 0;
    P.s_end = n;
    P.T = T;
    P.reject_mode = o->reject_mode;
    P.idx_v = o->idx_v - 1;
    P.idx_dh = o->idx_dh - 1;
    P.idx_L = o->idx_L - 1;
    P.is_quantize500 = o->is_quantize500;
    P.n_layers = o->n_layers;
    P.max_attempts = o->max_attempts > 0 ? o->max_attempts : 65534;
    if (P.max_attempts > 65534) P.max_attempts = 65534;   // `attempts` is uint16 and holds attempt + 1
    const int nv = H.n_initial;
    // bn_sample.m:45-50 preset validation
    for (int i = 0; i < nv; ++i) {
        const int32_t st = o->start[i];
        if (st < 0 || st > H.r_initial[i]) fail(EMB_E_ARG, "start: preset bin out of range");
        P.start[i] = (uint8_t)st;
    }
    for (int i = 0; i < nv; ++i) {
        if (!P.start[i]) continue;
        for (int p : H.T_initial[i].parents)
            if (!P.start[p]) fail(EMB_E_ARG, "Attempt to preset a dependent variable");
    }
    if (P.reject_mode == EMB_REJECT_UNCOR) {
        if (P.idx_v < 0 || P.idx_v >= nv || P.idx_dh < 0 || P.idx_dh >= nv)
            fail(EMB_E_ARG, "dynvar:empty: idx_v / idx_dh must name initial variables");
        if (P.n_layers > 0 || P.is_quantize500) {
            if (P.idx_L < 0 || P.idx_L >= nv) fail(EMB_E_ARG, "layers/isQuantize500 need idx_L");
            if (P.n_layers > 0) {
                if (P.n_layers > 8 || P.n_layers < H.r_initial[P.idx_L])
                    fail(EMB_E_ARG, "layers must have one row per altitude-layer bin (max 8)");
                if (!H.boundaries[P.idx_L].empty())
                    fail(EMB_E_ARG, "layers need the altitude layer to be sampled as a bin index "
                                              "(isOverwriteZeroBoundaries=true)");
            }
        }
        std::memcpy(P.layers, o->layers, sizeof(P.layers));
    } else if (P.reject_mode == EMB_REJECT_BOX) {
        for (int i = 0; i < nv; ++i) {
            P.box_lo[i] = o->box_lo[i];
            P.box_hi[i] = o->box_hi[i];
        }
    } else if (P.reject_mode != EMB_REJECT_NONE) {
        fail(EMB_E_ARG, "unknown reject_mode");
    }
}


// ------------------------------------------------------------------------------------------------
bool named_dyn_limits(const char* ac_type, TermLimits& out) {
    std::string t(ac_type ? ac_type : "");
    for (auto& c : t) c = (char)std::toupper((unsigned char)c);
    // minVel_ft_s, maxVel_ft_s, maxTurnRate_deg_s, maxAltitude_ft, maxVertRate_ft_s (getDynamicLimits.m:14-62)
    if (t == "GENERIC") out = TermLimits{50.0, 506.0, 12.0, 5000.0, 6000.0 / 60.0};
    else if (t == "RTCA228_A1") out = TermLimits{169.0, 491.0, 1.5, 5000.0, 2500.0 / 60.0};
    else if (t == "RTCA228_A2") out = TermLimits{68.0, 338.0, 3.0, 5000.0, 1500.0 / 60.0};
    else if (t == "RTCA228_A3") out = TermLimits{68.0, 186.0, 7.0, 5000.0, 500.0 / 60.0};
    else if (t == "TEST") out = TermLimits{68.0, 186.0, 7.0, 1200.0, 500.0 / 60.0};
    else return false;
    return true;
}

// min{s >= 0 : sqrt(s) >= c} for c > 0: sqrt is monotone and correctly rounded, so "norm >= c" is exactly "x*x + y*y >= s"
static double sq_threshold(double c) {
    const double inf = std::numeric_limits<double>::infinity();
    if (!(c > 0.0)) return 0.0;
    if (std::isinf(c)) return inf;
    double s = c * c;
    if (std::isinf(s)) return inf;
    while (s > 0.0 && std::sqrt(std::nextafter(s, 0.0)) >= c) s = std::nextafter(s, 0.0);
    while (std::sqrt(s) < c) s = std::nextafter(s, inf);
    return s;
}

void make_term_model(const HostModel& H, const TermLimits& lim, TermModel& M, double* cuts) {
    std::memset(&M, 0, sizeof(M));
    auto find = [&](const char* name) {
        const std::string q = std::string("\"") + name + "\"";
        for (int i = 0; i < H.n_initial; ++i)
            if (H.labels_initial[i] == q) return i;
        fail(EMB_E_MODEL, std::string("createEncounter: trajectory model has no variable ") + q);
        return -1;
    };
    if (H.n_initial != 6 || !H.has_transition)
        fail(EMB_E_MODEL, "createEncounter: a trajectory model has six initial variables and a transition network");
    find("intent");
    M.i_dist = find("distance");
    M.i_bear = find("bearing");
    if (find("heading") != 3 || find("altitude") != 4 || find("speed") != 5)                 // createEncounter.m:107-109
        fail(EMB_E_MODEL, "createEncounter: variables 4-6 must be \"heading\", \"altitude\", \"speed\"");
    if (H.temporal_map.size() != 3 || H.temporal_map[0].first != 3 || H.temporal_map[1].first != 4 ||
        H.temporal_map[2].first != 5)
        fail(EMB_E_MODEL, "createEncounter: the dynamic variables must be heading, altitude and speed");
    if (H.thr_transition.size() >= (1u << 26))
        fail(EMB_E_LIMIT, "createEncounter: transition table of a trajectory model exceeds 2^26 words");
    if (H.is_dynvar_depend)
        fail(EMB_E_MODEL, "createEncounter: trajectory models have no dynamic->dynamic edge (dbn_sample.m:95-166 branch)");
    if (H.prior_transition.kind != EMB_PRIOR_STAY || H.prior_transition.value != 1.0)
        fail(EMB_E_ARG, "createEncounter: set the stay prior first, emb_set_prior(m, 1, EMB_PRIOR_STAY, 1.0) "
                        "(setTransitionPriors, createEncounter.m:129)");
    if (H.prior_initial.kind != EMB_PRIOR_CONSTANT || H.prior_initial.value != 0.0)
        fail(EMB_E_ARG, "createEncounter: the initial prior must be 0 (createEncounter.m:128)");
    for (int d = 0; d < 3; ++d) {
        const Node& nd = H.dev.dyn[d];
        M.off[d] = nd.off;
        M.rp[d] = (uint32_t)nd.rp;
        for (int p = 0; p < nd.np; ++p) {
            if (nd.par[p] >= 6) fail(EMB_E_MODEL, "createEncounter: parent outside the initial variables");
            M.stride[d][nd.par[p]] = nd.stride_rp[p];
        }
    }
    for (int i = 0; i < 6; ++i) {
        M.edge_off[i] = H.dev.edge_off[i];
        M.r[i] = H.r_initial[i];
    }
    for (int i : {3, 4, 5})
        if (H.boundaries[i].empty()) fail(EMB_E_MODEL, "createEncounter: heading, altitude and speed need boundaries");
    // :120  discreteValidAlt = 1:find(edges <= maxAltitude_ft, 1, 'last')
    const auto& ea = H.boundaries[4];
    M.alt_hi = 0;
    for (size_t j = 0; j < ea.size(); ++j)
        if (ea[j] <= lim.maxAlt) M.alt_hi = (int32_t)j + 1;
    // :123-125  s = find((edges >= minVel) == false, 1, 'last'); e = find(edges <= maxVel, 1, 'last'); s:e
    const auto& es = H.boundaries[5];
    int s1 = 0, e1 = 0;
    for (size_t j = 0; j < es.size(); ++j) {
        if (!(es[j] >= lim.minVel)) s1 = (int)j + 1;
        if (es[j] <= lim.maxVel) e1 = (int)j + 1;
    }
    if (s1 == 0 || e1 == 0) {   // an empty find() makes s:e empty
        M.spd_lo = 1;
        M.spd_hi = 0;
    } else {
        M.spd_lo = s1;
        M.spd_hi = e1;
    }
    // tests on d_nm as tests on x*x + y*y (emb_terminal.cuh: TC_DIST2)
    M.dist_max_sq = sq_threshold(std::nextafter(H.bounds_initial[M.i_dist].second, std::numeric_limits<double>::infinity()));
    M.quarter_sq = sq_threshold(std::nextafter(0.25, 1.0));
    // cutpoint tables (emb_terminal.cuh: term_cell)
    const double inf = std::numeric_limits<double>::infinity();
    const int var_of[TERM_NCUT] = {M.i_dist, M.i_bear, 3, 4, 5};
    for (int t = 0; t < TERM_NCUT; ++t) {
        const int i = var_of[t], r = H.r_initial[i];
        if (r > TERM_CUT_MAX)
            fail(EMB_E_LIMIT, "createEncounter: a trajectory model variable has more than 64 bins");
        double* row = cuts ? cuts + t * TERM_CUT_MAX : nullptr;
        if (!row) continue;
        for (int j = 0; j < TERM_CUT_MAX; ++j) row[j] = inf;
        const auto& e = H.boundaries[i];
        for (int j = 1; j < r; ++j) {
            const double c = e.empty() ? (double)(j + 1) : e[(size_t)j];   // no boundaries: cutpoints 2..r (em_read.m:128-136)
            double v = c;
            if (t == TC_DIST2) {
                v = c <= 0.0 ? -inf : sq_threshold(c);                     // a norm is never negative
            } else if (t == TC_BEAR) {                                      // bearings live in [0, 360)
                if (c <= 0.0) v = -inf;                                     // every bearing is >= this cutpoint
                else if (c >= 360.0) v = inf;                               // none is
                else {
                    double sn, cs;
                    sincosd(c, sn, cs);
                    v = pseudo_angle(cs, sn);
                }
            }
            row[j - 1] = v;
        }
    }
}

}  // namespace emb
