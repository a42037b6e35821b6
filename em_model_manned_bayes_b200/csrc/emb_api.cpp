// emb_api.cpp -- the C ABI of libemb200.so (include/emb200.h).  No torch, no C++ types across the
// boundary, no exceptions escape.  There is deliberately no CPU sampling path in this library.
#include <cuda_runtime_api.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/emb200.h"
#include "emb_integrate.cuh"
#include "emb_launch.h"
#include "emb_loglik.cuh"
#include "emb_model.h"

using emb::DevModel;
using emb::HostModel;

struct emb_model {
    std::unique_ptr<HostModel> h;
};

namespace {

thread_local std::string g_err;

int set_err(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define EMB_TRY try {
#define EMB_CATCH                                                        \
    }                                                                    \
    catch (const emb::Error& e) { return set_err(e.code, e.msg); }       \
    catch (const std::bad_alloc&) { return set_err(EMB_E_LIMIT, "out of host memory"); } \
    catch (const std::exception& e) { return set_err(EMB_E_ARG, e.what()); }

int cuda_fail(cudaError_t e, const char* what) {
    return set_err(EMB_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                          \
    do {                                                  \
        cudaError_t e__ = (call);                         \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// Upload (or refresh after emb_set_prior) the packed tables of a model to `device`.
int ensure_device(const HostModel& H, int device, DevModel& D) {
    std::lock_guard<std::mutex> lk(H.mu);
    auto& c = H.device_copies[device];
    if (c.version != H.version) {
        if (c.thr_initial) cudaFree(c.thr_initial);
        if (c.thr_transition) cudaFree(c.thr_transition);
        if (c.edges) cudaFree(c.edges);
        if (c.dd32) cudaFree(c.dd32);
        if (c.logp_initial) cudaFree(c.logp_initial);
        if (c.logp_transition) cudaFree(c.logp_transition);
        c.logp_initial = c.logp_transition = nullptr;
        c.logp_ok = false;
        c.thr_initial = c.thr_transition = nullptr;
        c.edges = nullptr;
        c.dd32 = nullptr;
        auto up = [&](const void* src, size_t bytes, void** dst) -> int {
            *dst = nullptr;
            if (!bytes) return 0;
            CU(cudaMalloc(dst, bytes));
            CU(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
            return 0;
        };
        int rc;
        if ((rc = up(H.thr_initial.data(), H.thr_initial.size() * 4, (void**)&c.thr_initial))) return rc;
        if ((rc = up(H.thr_transition.data(), H.thr_transition.size() * 4, (void**)&c.thr_transition))) return rc;
        if ((rc = up(H.edges.data(), H.edges.size() * 8, (void**)&c.edges))) return rc;
        if ((rc = up(H.dd32.data(), H.dd32.size() * 4, (void**)&c.dd32))) return rc;
        c.version = H.version;
    }
    D = H.dev;
    D.thr_init = c.thr_initial;
    D.thr_trans = c.thr_transition;
    D.edges = c.edges;
    D.dd32 = c.dd32;
    D.logp_init = D.logp_trans = nullptr;
    return 0;
}

// ensure_device plus the scoring tables, uploaded on the first scoring call so that sampling-only callers never hold them in HBM
int ensure_logp(const HostModel& H, int device, DevModel& D) {
    int rc = ensure_device(H, device, D);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(H.mu);
    auto& c = H.device_copies[device];
    if (!c.logp_ok) {
        for (auto* t : {&H.logp_initial, &H.logp_transition}) {
            double*& dst = t == &H.logp_initial ? c.logp_initial : c.logp_transition;
            if (t->empty()) continue;
            CU(cudaMalloc((void**)&dst, t->size() * 8));
            CU(cudaMemcpy(dst, t->data(), t->size() * 8, cudaMemcpyHostToDevice));
        }
        c.logp_ok = true;
    }
    D.logp_init = c.logp_initial;
    D.logp_trans = c.logp_transition;
    return 0;
}

int pick_device(const emb_sample_opts* o, int& device, bool allow_async = false) {
    if ((o->mem & ~0xFF) && !(allow_async && (o->mem & ~0xFF) == EMB_MEM_ASYNC && (o->mem & 0xFF) == EMB_MEM_DEVICE))
        return set_err(EMB_E_ARG, "emb_sample_opts.mem: EMB_MEM_ASYNC goes with EMB_MEM_DEVICE, in emb_sample_tracks and emb_sample_initial only");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
        return set_err(EMB_E_CUDA, std::string("no CUDA device available (libemb200 has no CPU path): ") +
                                       (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    device = o->device;
    if (device < 0) CU(cudaGetDevice(&device));
    if (device >= count) return set_err(EMB_E_ARG, "device ordinal out of range");
    CU(cudaSetDevice(device));
    return 0;
}

// EMB_MEM_ASYNC launches report an exhausted rejection loop through one persistent word per device (read by emb_async_status)
std::mutex g_async_mu;
std::map<int, int32_t*> g_async_status;
int async_status_word(int device, int32_t** out) {
    std::lock_guard<std::mutex> lk(g_async_mu);
    auto it = g_async_status.find(device);
    if (it == g_async_status.end()) {
        int32_t* p = nullptr;
        CU(cudaMalloc((void**)&p, 4));
        CU(cudaMemset(p, 0, 4));
        it = g_async_status.emplace(device, p).first;
    }
    *out = it->second;
    return 0;
}

// Device-side staging for host-memory callers.
// Per-call temporaries (staging buffers, counts, event rows) come from the device's stream-ordered memory pool with an
// unlimited release threshold: repeated calls reuse the same memory instead of paying cudaMalloc/cudaFree (several ms per GB,
// and an implicit device synchronisation) inside every call.  Model tables stay plain cudaMalloc.
cudaError_t tmp_alloc(void** p, size_t bytes, cudaStream_t st) {
    static thread_local int configured_for = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (configured_for != dev) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        configured_for = dev;
    }
    return cudaMallocAsync(p, bytes, st);
}
// Temporaries die when an entry point returns.  On the normal path every stream that touched them has been synchronised;
// on an early error return a kernel may still be running on the caller's (possibly non-blocking) stream, so the free is
// stream-ordered on THAT stream (the legacy stream would not wait for a non-blocking one); the second stream of the event
// pipeline is drained by its owner (Guard) before the buffers it reads are released.
thread_local cudaStream_t g_call_stream = nullptr;   // the caller's stream of the entry point running on this thread
void tmp_free(void* p) {
    if (p) cudaFreeAsync(p, g_call_stream);
}

struct Staged {
    void* host = nullptr;
    void* dev = nullptr;
    size_t bytes = 0;
    bool owned = false;
};
struct Stager {
    int mem;
    cudaStream_t stream;
    std::vector<Staged> items;
    ~Stager() {
        for (auto& s : items)
            if (s.owned && s.dev) tmp_free(s.dev);
    }
    // returns the device pointer to use for a caller buffer (nullptr stays nullptr)
    int out(void* user, size_t bytes, bool zero, void** dev) {
        *dev = nullptr;
        if (!user || !bytes) return 0;
        if (mem == EMB_MEM_DEVICE) {
            *dev = user;
            return 0;
        }
        Staged s;
        s.host = user;
        s.bytes = bytes;
        s.owned = true;
        CU(tmp_alloc(&s.dev, bytes, stream));
        if (zero) CU(cudaMemcpyAsync(s.dev, user, bytes, cudaMemcpyHostToDevice, stream));  // accumulate (+=) semantics
        items.push_back(s);
        *dev = s.dev;
        return 0;
    }
    // device copy of a caller INPUT buffer (not copied back)
    int in(const void* user, size_t bytes, const void** dev) {
        *dev = nullptr;
        if (!user || !bytes) return 0;
        if (mem == EMB_MEM_DEVICE) {
            *dev = user;
            return 0;
        }
        Staged s;
        s.bytes = bytes;
        s.owned = true;
        CU(tmp_alloc(&s.dev, bytes, stream));
        CU(cudaMemcpyAsync(s.dev, user, bytes, cudaMemcpyHostToDevice, stream));
        items.push_back(s);
        *dev = s.dev;
        return 0;
    }
    int finish() {
        for (auto& s : items)
            if (s.host) CU(cudaMemcpyAsync(s.host, s.dev, s.bytes, cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        return 0;
    }
};

// per-sample presets of emb_sample_opts -> SampleParams (device pointer, one row of n per initial variable)
int stage_start(Stager& sg, const emb_sample_opts* opts, const HostModel& H, int64_t n, emb::SampleParams& P) {
    P.start_ps = nullptr;
    P.start_stride = n;
    if (!opts->start_per_sample) return 0;
    const void* d = nullptr;
    int rc = sg.in(opts->start_per_sample, (size_t)n * (size_t)H.n_initial, &d);
    if (rc) return rc;
    P.start_ps = (const int8_t*)d;
    return 0;
}
// the device status word of the sampling kernels: 1 = rejection loop exhausted, 2 = invalid per-sample preset
int status_error(int32_t status) {
    if (status == 2)
        return set_err(EMB_E_ARG, "Attempt to preset a dependent variable (or a preset bin out of range) in start_per_sample");
    if (status) return set_err(EMB_E_REJECT, "a sample exhausted max_attempts in the rejection loop");
    return 0;
}

template <class T>
int64_t copy_out(const std::vector<T>& v, T* buf, int64_t cap) {
    if (buf) std::memcpy(buf, v.data(), sizeof(T) * (size_t)std::min<int64_t>(cap, (int64_t)v.size()));
    return (int64_t)v.size();
}

}  // namespace

// =================================================================================================
extern "C" {

int emb_abi_version(void) { return EMB_ABI_VERSION; }
const char* emb_last_error(void) { return g_err.c_str(); }
int64_t emb_launch_count(void) { return emb::g_launch_count.load(); }
void emb_debug_force_generic(int on) { emb::g_force_generic = on; }
int emb_debug_last_kernel_fast(void) { return emb::g_last_kernel_fast; }

int emb_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) return 0;
    return c;
}

int emb_host_alloc(void** p, int64_t bytes) {
    CU(cudaMallocHost(p, (size_t)bytes));
    return 0;
}
int emb_async_status(int device) {
    int dev = device;
    if (dev < 0) CU(cudaGetDevice(&dev));
    CU(cudaSetDevice(dev));
    CU(cudaDeviceSynchronize());
    int32_t* word = nullptr;
    int rc = async_status_word(dev, &word);
    if (rc) return rc;
    int32_t flag = 0;
    CU(cudaMemcpy(&flag, word, 4, cudaMemcpyDeviceToHost));
    if (flag) {
        CU(cudaMemset(word, 0, 4));
        return status_error(flag);
    }
    return 0;
}
int emb_trim_device_memory(int device) {
    int dev = device;
    if (dev < 0) CU(cudaGetDevice(&dev));
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, dev));
    CU(cudaDeviceSynchronize());
    CU(cudaMemPoolTrimTo(pool, 0));
    return 0;
}
int emb_host_free(void* p) {
    CU(cudaFreeHost(p));
    return 0;
}

uint32_t emb_rng_word(uint64_t seed, uint64_t sample, uint32_t attempt, uint32_t purpose, uint32_t index,
                      uint32_t sub, uint32_t lane) {
    return emb::keyed_word(seed, sample, attempt, purpose, index, sub, lane & 3u);
}

int emb_model_load(const char* path, int is_overwrite, const int32_t* idx_zero, int32_t n_idx, emb_model** out) {
    if (!path || !out) return set_err(EMB_E_ARG, "null argument");
    *out = nullptr;
    EMB_TRY
    std::unique_ptr<emb_model> m(new emb_model());
    m->h.reset(emb::load_model_file(path, is_overwrite != 0, idx_zero, idx_zero ? n_idx : 0));
    *out = m.release();
    return 0;
    EMB_CATCH
}

int emb_model_from_arrays(int32_t n_initial, const uint8_t* G_initial, const int32_t* r_initial,
                          const double* N_initial, int64_t len_N_initial, int32_t n_transition,
                          const uint8_t* G_transition, const int32_t* r_transition, const double* N_transition,
                          int64_t len_N_transition, const int32_t* temporal_map, int32_t n_temporal,
                          const double* boundaries, const int32_t* boundaries_len, const double* resample_rates,
                          emb_model** out) {
    if (!out || !G_initial || !r_initial || !N_initial || n_initial <= 0) return set_err(EMB_E_ARG, "null argument");
    *out = nullptr;
    EMB_TRY
    std::unique_ptr<emb_model> m(new emb_model());
    m->h.reset(new HostModel());
    HostModel& H = *m->h;
    H.n_initial = n_initial;
    H.G_initial.assign(G_initial, G_initial + (size_t)n_initial * n_initial);
    H.r_initial.assign(r_initial, r_initial + n_initial);
    for (int i = 0; i < n_initial; ++i) H.labels_initial.push_back("\"x" + std::to_string(i + 1) + "\"");
    auto fill = [&](const std::vector<uint8_t>& G, const std::vector<int32_t>& r, int n, int first, const double* x,
                    int64_t len, std::vector<emb::Table>& T, const char* what) {
        T.assign(n, emb::Table{});
        int64_t index = 0;
        for (int i = first; i < n; ++i) {
            emb::Table& t = T[i];
            t.r = r[i];
            t.q = 1;
            for (int p = 0; p < n; ++p)
                if (G[(size_t)p * n + i]) {
                    t.parents.push_back(p);
                    t.q *= r[p];
                }
            const int64_t cnt = (int64_t)t.r * t.q;
            if (index + cnt > len) throw emb::Error{EMB_E_ARG, std::string(what) + " is shorter than sum(r_i*q_i)"};
            t.N.assign(x + index, x + index + cnt);
            t.present = true;
            index += cnt;
        }
        if (index != len) throw emb::Error{EMB_E_ARG, std::string(what) + " is longer than sum(r_i*q_i)"};
    };
    fill(H.G_initial, H.r_initial, n_initial, 0, N_initial, len_N_initial, H.T_initial, "N_initial");
    if (n_transition > 0 && G_transition && r_transition && N_transition) {
        H.has_transition = true;
        H.n_transition = n_transition;
        H.G_transition.assign(G_transition, G_transition + (size_t)n_transition * n_transition);
        H.r_transition.assign(r_transition, r_transition + n_transition);
        for (int i = 0; i < n_transition; ++i) H.labels_transition.push_back("\"y" + std::to_string(i + 1) + "\"");
        fill(H.G_transition, H.r_transition, n_transition, n_initial, N_transition, len_N_transition, H.T_transition,
             "N_transition");
        if (!temporal_map || n_temporal <= 0) throw emb::Error{EMB_E_ARG, "temporal_map is required with a transition network"};
        for (int k = 0; k < n_temporal; ++k) {
            const int a = temporal_map[2 * k] - 1, b = temporal_map[2 * k + 1] - 1;
            if (a < 0 || a >= n_initial || b < n_initial || b >= n_transition)
                throw emb::Error{EMB_E_ARG, "temporal_map entry out of range"};
            H.temporal_map.push_back({a, b});
        }
        H.temporal_map_given = true;
    }
    H.boundaries.assign(n_initial, {});
    if (boundaries && boundaries_len) {
        const double* b = boundaries;
        for (int i = 0; i < n_initial; ++i) {
            H.boundaries[i].assign(b, b + boundaries_len[i]);
            b += boundaries_len[i];
        }
        H.has_boundaries = true;
    }
    if (resample_rates) H.resample_rates.assign(resample_rates, resample_rates + n_initial);
    H.derive();
    H.pack();
    *out = m.release();
    return 0;
    EMB_CATCH
}

void emb_model_free(emb_model* m) {
    if (!m) return;
    if (m->h) {
        for (auto& kv : m->h->device_copies) {
            int cur = 0;
            if (cudaGetDevice(&cur) == cudaSuccess && cudaSetDevice(kv.first) == cudaSuccess) {
                if (kv.second.thr_initial) cudaFree(kv.second.thr_initial);
                if (kv.second.thr_transition) cudaFree(kv.second.thr_transition);
                if (kv.second.edges) cudaFree(kv.second.edges);
                if (kv.second.dd32) cudaFree(kv.second.dd32);
                if (kv.second.logp_initial) cudaFree(kv.second.logp_initial);
                if (kv.second.logp_transition) cudaFree(kv.second.logp_transition);
                cudaSetDevice(cur);
            }
        }
    }
    delete m;
}

int emb_model_get_info(const emb_model* m, emb_model_info* info) {
    if (!m || !info) return set_err(EMB_E_ARG, "null argument");
    const HostModel& H = *m->h;
    std::memset(info, 0, sizeof(*info));
    info->n_initial = H.n_initial;
    info->n_transition = H.has_transition ? H.n_transition : 0;
    info->n_dyn = (int32_t)H.temporal_map.size();
    info->n_gated = (int32_t)H.gated.size();
    info->is_dynvar_depend = H.is_dynvar_depend ? 1 : 0;
    info->n_timevarying = (int32_t)H.timevarying.size();
    for (auto& t : H.T_initial) info->len_N_initial += (int64_t)t.N.size();
    for (auto& t : H.T_transition) info->len_N_transition += (int64_t)t.N.size();
    for (int i = 0; i < H.n_initial; ++i) {
        info->r_initial[i] = H.r_initial[i];
        info->order_initial[i] = H.order_initial[i] + 1;
        info->zero_bins[i] = H.zero_bins[i];
        info->boundaries_len[i] = (int32_t)H.boundaries[i].size();
        info->resample_rates[i] = H.resample_rates[i];
        info->bounds_initial[i][0] = H.bounds_initial[i].first;
        info->bounds_initial[i][1] = H.bounds_initial[i].second;
    }
    if (H.has_transition)
        for (int i = 0; i < H.n_transition; ++i) {
            info->r_transition[i] = H.r_transition[i];
            info->order_transition[i] = H.order_transition[i] + 1;
        }
    for (size_t k = 0; k < H.temporal_map.size(); ++k) {
        info->temporal_map[k][0] = H.temporal_map[k].first + 1;
        info->temporal_map[k][1] = H.temporal_map[k].second + 1;
    }
    for (size_t k = 0; k < H.timevarying.size(); ++k) info->timevarying_vars[k] = H.timevarying[k] + 1;
    return 0;
}

int64_t emb_model_get_labels(const emb_model* m, int which, char* buf, int64_t cap) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    const auto& L = which ? m->h->labels_transition : m->h->labels_initial;
    std::string s;
    for (size_t i = 0; i < L.size(); ++i) {
        if (i) s.push_back('\n');
        s += L[i];
    }
    if (buf && cap > 0) {
        const size_t k = std::min<size_t>((size_t)cap - 1, s.size());
        std::memcpy(buf, s.data(), k);
        buf[k] = 0;
    }
    return (int64_t)s.size() + 1;
}

int64_t emb_model_get_G(const emb_model* m, int which, uint8_t* buf, int64_t cap) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    return copy_out(which ? m->h->G_transition : m->h->G_initial, buf, cap);
}

int64_t emb_model_get_N(const emb_model* m, int which, double* buf, int64_t cap) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    std::vector<double> all;
    for (auto& t : (which ? m->h->T_transition : m->h->T_initial)) all.insert(all.end(), t.N.begin(), t.N.end());
    return copy_out(all, buf, cap);
}

int64_t emb_model_get_boundaries(const emb_model* m, double* buf, int64_t cap) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    std::vector<double> all;
    for (auto& b : m->h->boundaries) all.insert(all.end(), b.begin(), b.end());
    return copy_out(all, buf, cap);
}

int64_t emb_model_get_packed(const emb_model* m, int which, uint32_t* buf, int64_t cap) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    return copy_out(which ? m->h->thr_transition : m->h->thr_initial, buf, cap);
}

int emb_set_prior(emb_model* m, int which, int kind, double value) {
    if (!m) return set_err(EMB_E_ARG, "null argument");
    if (kind != EMB_PRIOR_CONSTANT && kind != EMB_PRIOR_DBE && kind != EMB_PRIOR_STAY)
        return set_err(EMB_E_ARG, "prior:unknown");
    if (kind == EMB_PRIOR_STAY && which == 0) return set_err(EMB_E_ARG, "stay prior applies to the transition network only");
    if (kind != EMB_PRIOR_DBE && !(value >= 0.0)) return set_err(EMB_E_ARG, "prior must be >= 0");
    EMB_TRY
    HostModel& H = *m->h;
    std::lock_guard<std::mutex> lk(H.mu);
    emb::PriorSpec old_i = H.prior_initial, old_t = H.prior_transition;
    (which ? H.prior_transition : H.prior_initial) = emb::PriorSpec{kind, value};
    try {
        H.pack();
    } catch (...) {
        H.prior_initial = old_i;
        H.prior_transition = old_t;
        H.pack();
        throw;
    }
    return 0;
    EMB_CATCH
}

void emb_sample_opts_init(emb_sample_opts* o) {
    std::memset(o, 0, sizeof(*o));
    o->device = -1;
    o->mem = EMB_MEM_HOST;
    for (int i = 0; i < EMB_MAX_VARS; ++i) {
        o->box_lo[i] = -1.0 / 0.0;
        o->box_hi[i] = 1.0 / 0.0;
    }
}

// values: double (values64) or float (values32), at most one of them
static int sample_initial_impl(const emb_model* m, const emb_rng* rng, int64_t n, const emb_sample_opts* opts, int8_t* bins,
                               double* values64, float* values32, uint16_t* attempts) {
    if (!m || !rng || !opts || n < 0) return set_err(EMB_E_ARG, "null or negative argument");
    const HostModel& H = *m->h;
    emb::SampleParams P;
    int rc = 0;
    try {
        emb::fill_params(H, rng->seed, rng->first_sample, n, 0, *opts, P);
    } catch (const emb::Error& e) {
        return set_err(e.code, e.msg);
    }
    if (n == 0) return 0;
    int device;
    if ((rc = pick_device(opts, device, true))) return rc;
    DevModel D;
    if ((rc = ensure_device(H, device, D))) return rc;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    const int tw = (int)H.thr_initial.size();
    auto launch = [&](int8_t* b, double* v64, float* v32, uint16_t* a, int32_t* word) {
        return v32 ? (cudaError_t)emb::launch_initial_f32(D, P, tw, b, v32, a, nullptr, word, st)
                   : (cudaError_t)emb::launch_initial(D, P, tw, b, v64, a, nullptr, word, st);
    };
    P.start_ps = opts->start_per_sample;   // device pointer in the enqueue-only path; staged below otherwise
    P.start_stride = n;
    if (opts->mem & EMB_MEM_ASYNC) {   // enqueue only (device buffers): see emb_sample_tracks
        int32_t* word = nullptr;
        if ((rc = async_status_word(device, &word))) return rc;
        const cudaError_t ea = launch(bins, values64, values32, attempts, word);
        return ea == cudaSuccess ? 0 : cuda_fail(ea, "launch k_initial");
    }
    Stager sg{opts->mem, st, {}};
    int8_t* d_bins;
    double* d_v64;
    float* d_v32;
    uint16_t* d_att;
    if ((rc = sg.out(bins, (size_t)n * H.n_initial, false, (void**)&d_bins))) return rc;
    if ((rc = sg.out(values64, (size_t)n * H.n_initial * 8, false, (void**)&d_v64))) return rc;
    if ((rc = sg.out(values32, (size_t)n * H.n_initial * 4, false, (void**)&d_v32))) return rc;
    if ((rc = sg.out(attempts, (size_t)n * 2, false, (void**)&d_att))) return rc;
    if ((rc = stage_start(sg, opts, H, n, P))) return rc;
    int32_t* d_status = nullptr;
    CU(tmp_alloc((void**)&d_status, 4, st));
    CU(cudaMemsetAsync(d_status, 0, 4, st));
    cudaError_t e = launch(d_bins, d_v64, d_v32, d_att, d_status);
    if (e != cudaSuccess) {
        tmp_free(d_status);
        return cuda_fail(e, "launch k_initial");
    }
    int32_t status = 0;
    e = cudaMemcpyAsync(&status, d_status, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    tmp_free(d_status);
    if (e != cudaSuccess) return cuda_fail(e, "k_initial");
    if ((rc = sg.finish())) return rc;
    return status_error(status);
}

int emb_sample_initial(const emb_model* m, const emb_rng* rng, int64_t n, const emb_sample_opts* opts, int8_t* bins,
                       double* values, uint16_t* attempts) {
    return sample_initial_impl(m, rng, n, opts, bins, values, nullptr, attempts);
}
int emb_sample_initial_f32(const emb_model* m, const emb_rng* rng, int64_t n, const emb_sample_opts* opts, int8_t* bins,
                           float* values, uint16_t* attempts) {
    if (!values) return set_err(EMB_E_ARG, "emb_sample_initial_f32: values must not be null (use emb_sample_initial for bins only)");
    return sample_initial_impl(m, rng, n, opts, bins, nullptr, values, attempts);
}

int64_t emb_tracks_bins_len(const emb_model* m, int64_t n, int32_t T) {
    if (!m || n < 0 || T < 0) return 0;
    const int64_t nch4 = (T + 3) / 4;
    return (int64_t)m->h->temporal_map.size() * nch4 * emb::num_tiles(n) * emb::TRACK_TILE * 4;
}
int64_t emb_tracks_values_len(const emb_model* m, int64_t n, int32_t T) {
    if (!m || n < 0 || T < 0) return 0;
    const int64_t nch4 = (T + 3) / 4;
    return (int64_t)m->h->timevarying.size() * nch4 * emb::num_tiles(n) * emb::TRACK_TILE * 4;
}

int emb_sample_tracks(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                      const emb_track_out* out) {
    if (!m || !rng || !opts || !out || n < 0 || T < 1) return set_err(EMB_E_ARG, "null or out-of-range argument");
    const HostModel& H = *m->h;
    if (!H.has_transition || H.temporal_map.empty())
        return set_err(EMB_E_ARG, "dynvar:empty: model has no transition network");
    if ((int64_t)T * (int64_t)H.gated.size() >= (1ll << 33))
        return set_err(EMB_E_LIMIT, "T too large for the 32-bit stream index");
    emb::SampleParams P;
    int rc = 0;
    try {
        emb::fill_params(H, rng->seed, rng->first_sample, n, T, *opts, P);
    } catch (const emb::Error& e) {
        return set_err(e.code, e.msg);
    }
    if (n == 0) return 0;
    int device;
    if ((rc = pick_device(opts, device, true))) return rc;
    DevModel D;
    if ((rc = ensure_device(H, device, D))) return rc;
    if (opts->correct_dbn) D.fast = 0;      // parents re-evaluated every second (emb_sample_opts::correct_dbn)
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    const bool async = (opts->mem & EMB_MEM_ASYNC) != 0;
    Stager sg{opts->mem & 0xFF, st, {}};
    emb::TrackOut O{};
    const size_t ni = (size_t)H.n_initial;
    if ((rc = sg.out(out->bins, (size_t)emb_tracks_bins_len(m, n, T), false, (void**)&O.bins))) return rc;
    if ((rc = sg.out(out->values, (size_t)emb_tracks_values_len(m, n, T) * 4, false, (void**)&O.values))) return rc;
    if ((rc = sg.out(out->init_bins, (size_t)n * ni, false, (void**)&O.init_bins))) return rc;
    if ((rc = sg.out(out->init_values, (size_t)n * ni * 8, false, (void**)&O.init_values))) return rc;
    if ((rc = sg.out(out->attempts, (size_t)n * 2, false, (void**)&O.attempts))) return rc;
    if (out->hist_initial || out->hist_transition) {   // the histograms have 64 counters per variable
        for (int i = 0; i < H.n_initial; ++i)
            if (H.r_initial[i] > 64) return set_err(EMB_E_LIMIT, "verification histograms hold 64 bins per variable; this model has a variable with more");
    }
    if ((rc = sg.out(out->hist_initial, ni * 64 * 8, true, (void**)&O.hist_initial))) return rc;
    if ((rc = sg.out(out->hist_transition, H.temporal_map.size() * 64 * 8, true, (void**)&O.hist_transition))) return rc;
    if ((rc = stage_start(sg, opts, H, n, P))) return rc;
    if (async) {   // enqueue only: no host round trip between consecutive passes; emb_async_status collects the flag
        if ((rc = async_status_word(device, &O.status))) return rc;
        const cudaError_t ea = (cudaError_t)emb::launch_tracks(D, P, O, st);
        return ea == cudaSuccess ? 0 : cuda_fail(ea, "launch k_tracks");
    }
    CU(tmp_alloc((void**)&O.status, 4, st));
    CU(cudaMemsetAsync(O.status, 0, 4, st));
    cudaError_t e = (cudaError_t)emb::launch_tracks(D, P, O, st);
    if (e != cudaSuccess) {
        tmp_free(O.status);
        return cuda_fail(e, "launch k_tracks");
    }
    int32_t status = 0;
    e = cudaMemcpyAsync(&status, O.status, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    tmp_free(O.status);
    if (e != cudaSuccess) return cuda_fail(e, "k_tracks");
    if ((rc = sg.finish())) return rc;
    return status_error(status);
}

// EMB200_TRACE=1: host-side phase times of emb_sample_track_events on stderr (diagnostics for the e2e number)
struct PhaseTrace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    PhaseTrace() : on(std::getenv("EMB200_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[emb200] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// Both event entry points.  The write pass always produces packed rows on the device (emb_device.cuh: pack_event_word);
// `events` != nullptr: the 8-byte emb_event rows, expanded on the device before they leave it;
// `words` / `dts` != nullptr: the packed rows themselves (5 bytes per row over PCIe instead of 8).
static int sample_events_impl(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                              int64_t capacity, emb_event* events, uint32_t* words, uint8_t* dts, int64_t* offsets,
                              const emb_track_out* init, int64_t* total_rows) {
    const bool packed = events == nullptr;
    if (!m || !rng || !opts || !offsets || n < 0 || T < 1 || capacity < 0 || (capacity > 0 && packed && (!words || !dts)))
        return set_err(EMB_E_ARG, "null or out-of-range argument");
    if (init && (init->bins || init->values || init->hist_initial || init->hist_transition))
        return set_err(EMB_E_ARG, "emb_sample_track_events: dense outputs and histograms belong to emb_sample_tracks");
    const HostModel& H = *m->h;
    if (!H.has_transition || H.temporal_map.empty())
        return set_err(EMB_E_ARG, "dynvar:empty: model has no transition network");
    int max_bins = 0;
    for (int v : H.gated) max_bins = std::max(max_bins, (int)H.r_initial[v]);
    emb::EventFormat fm{};
    if (!emb::event_format_for((int)H.gated.size(), max_bins, T, fm))
        return set_err(EMB_E_LIMIT, "event rows need <= 15 time-varying variables with <= 16 bins each and T <= 65535");
    if (packed && (fm.gord_bits != 3 || fm.dt_bytes != 1))
        return set_err(EMB_E_LIMIT, "packed event rows need <= 7 time-varying variables and T <= 1023 (use emb_sample_track_events)");
    emb::SampleParams P;
    int rc = 0;
    try {
        emb::fill_params(H, rng->seed, rng->first_sample, n, T, *opts, P);
    } catch (const emb::Error& e) {
        return set_err(e.code, e.msg);
    }
    int device;
    if ((rc = pick_device(opts, device))) return rc;
    DevModel D;
    if ((rc = ensure_device(H, device, D))) return rc;
    if (opts->correct_dbn) D.fast = 0;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    if (total_rows) *total_rows = 0;
    if (n == 0) {
        const int64_t zero = 0;
        if (opts->mem == EMB_MEM_DEVICE) CU(cudaMemcpyAsync(offsets, &zero, 8, cudaMemcpyHostToDevice, st));
        else offsets[0] = 0;
        return 0;
    }
    PhaseTrace tr;
    Stager sg{opts->mem, st, {}};
    const size_t ni = (size_t)H.n_initial;
    emb::TrackOut O{};
    O.ev_gord_bits = fm.gord_bits;
    O.ev_dt_bytes = fm.dt_bytes;
    long long* d_off = nullptr;
    if ((rc = sg.out(offsets, (size_t)(n + 1) * 8, false, (void**)&d_off))) return rc;
    if (init) {
        if ((rc = sg.out(init->init_bins, (size_t)n * ni, false, (void**)&O.init_bins))) return rc;
        if ((rc = sg.out(init->init_values, (size_t)n * ni * 8, false, (void**)&O.init_values))) return rc;
        if ((rc = sg.out(init->attempts, (size_t)n * 2, false, (void**)&O.attempts))) return rc;
    }
    if ((rc = stage_start(sg, opts, H, n, P))) return rc;
    struct Scratch {
        void* p = nullptr;
        ~Scratch() { tmp_free(p); }
    } counts, status, tiles, pw, pd;
    CU(tmp_alloc(&counts.p, (size_t)n * 4, st));
    CU(tmp_alloc(&tiles.p, (size_t)emb::scan_scratch_len(n) * 8, st));
    CU(tmp_alloc(&status.p, 4, st));
    CU(cudaMemsetAsync(status.p, 0, 4, st));
    O.status = (int32_t*)status.p;
    const bool host = (opts->mem & 0xFF) == EMB_MEM_HOST;
    const bool pipelined = host && n >= 8192;
    if (!pipelined) {
        // pass 1: rows per track (also writes the per-track initial outputs), then the prefix sum
        O.ev_counts = (uint32_t*)counts.p;
        cudaError_t e = (cudaError_t)emb::launch_tracks(D, P, O, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_tracks (event count)");
        e = (cudaError_t)emb::launch_scan_counts((const uint32_t*)counts.p, d_off, n, (long long*)tiles.p, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_scan_counts");
        long long total = 0;
        int32_t flag = 0;
        CU(cudaMemcpyAsync(&total, d_off + n, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&flag, status.p, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        tr.mark("alloc + count pass + scan");
        if (total_rows) *total_rows = total;
        if (flag) return status_error(flag);
        if (total > capacity) {
            if ((rc = sg.finish())) return rc;   // offsets and the initial outputs are valid
            return set_err(EMB_E_LIMIT, "event buffer too small: " + std::to_string(total) + " rows needed");
        }
        // pass 2: write the packed rows (the keyed stream reproduces pass 1 exactly)
        O.ev_counts = nullptr;
        O.init_bins = nullptr;
        O.init_values = nullptr;
        O.attempts = nullptr;
        uint32_t* d_words = nullptr;
        uint8_t* d_dts = nullptr;
        if (packed) {
            if ((rc = sg.out(words, (size_t)total * 4, false, (void**)&d_words))) return rc;
            if ((rc = sg.out(dts, (size_t)total, false, (void**)&d_dts))) return rc;
        } else {
            CU(tmp_alloc(&pw.p, (size_t)std::max<long long>(total, 1) * 4, st));
            CU(tmp_alloc(&pd.p, (size_t)std::max<long long>(total, 1) * fm.dt_bytes, st));
            d_words = (uint32_t*)pw.p;
            d_dts = (uint8_t*)pd.p;
        }
        O.ev_offsets = d_off;
        O.ev_words = d_words;
        O.ev_dts = d_dts;
        e = (cudaError_t)emb::launch_tracks(D, P, O, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_tracks (event write)");
        if (!packed) {
            uint2* d_ev = nullptr;
            if ((rc = sg.out(events, (size_t)total * 8, false, (void**)&d_ev))) return rc;
            e = (cudaError_t)emb::launch_expand_events(D, d_words, d_dts, d_ev, 0, total, fm, st);
            if (e != cudaSuccess) return cuda_fail(e, "launch k_expand_events");
        }
        CU(cudaStreamSynchronize(st));
        return sg.finish();
    }
    // Host-memory caller, large batch: the tracks go through in chunks, each chunk = count pass -> prefix sum (carrying the
    // rows of the chunks before it) -> write pass (-> expansion) on the caller's stream, while a second stream copies the rows
    // of the finished chunks to the host (rows of a track range are contiguous: [offsets[a], offsets[b])).  Only the first
    // chunk's count pass is not hidden behind a copy.
    struct Guard {
        void* rows = nullptr;       // 8-byte rows (legacy entry point only)
        cudaStream_t copy = nullptr;
        cudaEvent_t done[16] = {};
        ~Guard() {
            for (auto& d : done) if (d) cudaEventDestroy(d);
            if (copy) {
                cudaStreamSynchronize(copy);
                cudaStreamDestroy(copy);
            }
            tmp_free(rows);
        }
    } g;
    if (capacity > 0) {
        CU(tmp_alloc(&pw.p, (size_t)capacity * 4, st));
        CU(tmp_alloc(&pd.p, (size_t)capacity * fm.dt_bytes, st));
        if (!packed) CU(tmp_alloc(&g.rows, (size_t)capacity * 8, st));
    }
    CU(cudaStreamCreateWithFlags(&g.copy, cudaStreamNonBlocking));
    CU(cudaMemsetAsync(d_off, 0, 8, st));                 // carry of the first chunk
    const int chunks = 8;
    long long total = 0;
    bool overflow = false;
    static thread_local long long* pub = nullptr;         // mapped pinned host memory, 2 words per chunk, kept for the thread
    if (!pub) CU(cudaHostAlloc((void**)&pub, sizeof(long long) * 2 * 16, cudaHostAllocMapped | cudaHostAllocPortable));
    for (int c = 0; c < chunks; ++c) {
        const int64_t a = n * c / chunks, b = n * (c + 1) / chunks;
        if (b <= a) continue;
        emb::SampleParams Pc = P;
        Pc.first_sample = P.first_sample + (uint64_t)a;
        Pc.n = b - a;
        Pc.s_begin = 0;
        Pc.s_end = b - a;
        if (P.start_ps) Pc.start_ps = P.start_ps + a;     // rows stay n apart (start_stride)
        emb::TrackOut Oc = O;                             // count pass of the chunk: also its per-track initial outputs
        Oc.init_stride = n;
        if (O.init_bins) Oc.init_bins = O.init_bins + a;
        if (O.init_values) Oc.init_values = O.init_values + a;
        if (O.attempts) Oc.attempts = O.attempts + a;
        Oc.ev_counts = (uint32_t*)counts.p + a;
        cudaError_t e = (cudaError_t)emb::launch_tracks(D, Pc, Oc, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_tracks (event count)");
        e = (cudaError_t)emb::launch_scan_counts((const uint32_t*)counts.p + a, d_off + a, b - a, (long long*)tiles.p, st, d_off + a);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_scan_counts");
        // the chunk's running total and the rejection flag reach the host through mapped memory (an SM store): a cudaMemcpy
        // would queue on the copy engine behind the previous chunk's rows and serialise the pipeline
        e = (cudaError_t)emb::launch_publish(d_off + b, (const int32_t*)status.p, pub + 2 * c, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_publish");
        CU(cudaStreamSynchronize(st));
        const long long r0 = total, r1 = pub[2 * c];
        const int32_t flag = (int32_t)pub[2 * c + 1];
        if (c == 0) tr.mark("first chunk: count + scan");
        if (flag) {
            CU(cudaStreamSynchronize(g.copy));
            return status_error(flag);
        }
        total = r1;
        if (total > capacity) overflow = true;            // keep counting: the caller learns how many rows are needed
        if (overflow || r1 == r0) continue;
        emb::TrackOut Ow{};                               // write pass of the chunk (the keyed stream reproduces the count pass)
        Ow.status = O.status;
        Ow.ev_offsets = d_off + a;
        Ow.ev_words = (uint32_t*)pw.p;
        Ow.ev_dts = (uint8_t*)pd.p;
        Ow.ev_gord_bits = fm.gord_bits;
        Ow.ev_dt_bytes = fm.dt_bytes;
        e = (cudaError_t)emb::launch_tracks(D, Pc, Ow, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch k_tracks (event write)");
        if (!packed) {
            e = (cudaError_t)emb::launch_expand_events(D, (const uint32_t*)pw.p, (const uint8_t*)pd.p, g.rows, r0, r1 - r0, fm, st);
            if (e != cudaSuccess) return cuda_fail(e, "launch k_expand_events");
        }
        CU(cudaEventCreateWithFlags(&g.done[c], cudaEventDisableTiming));
        CU(cudaEventRecord(g.done[c], st));
        CU(cudaStreamWaitEvent(g.copy, g.done[c], 0));
        if (packed) {
            CU(cudaMemcpyAsync(words + r0, (const uint32_t*)pw.p + r0, (size_t)(r1 - r0) * 4, cudaMemcpyDeviceToHost, g.copy));
            CU(cudaMemcpyAsync(dts + r0, (const uint8_t*)pd.p + r0, (size_t)(r1 - r0), cudaMemcpyDeviceToHost, g.copy));
        } else {
            CU(cudaMemcpyAsync(events + r0, (const char*)g.rows + (size_t)r0 * 8, (size_t)(r1 - r0) * 8, cudaMemcpyDeviceToHost, g.copy));
        }
    }
    tr.mark("chunks enqueued");
    if (total_rows) *total_rows = total;
    if ((rc = sg.finish())) return rc;          // offsets and per-track outputs, on the caller's stream
    tr.mark("finish (offsets, inits D2H)");
    CU(cudaStreamSynchronize(g.copy));
    tr.mark("rows D2H drained");
    if (overflow) return set_err(EMB_E_LIMIT, "event buffer too small: " + std::to_string(total) + " rows needed");
    return 0;
}

int emb_sample_track_events(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                            int64_t capacity, emb_event* events, int64_t* offsets, const emb_track_out* init,
                            int64_t* total_rows) {
    if (capacity > 0 && !events) return set_err(EMB_E_ARG, "null or out-of-range argument");
    emb_event dummy;
    return sample_events_impl(m, rng, n, T, opts, capacity, events ? events : &dummy, nullptr, nullptr, offsets, init, total_rows);
}

int emb_sample_track_events_packed(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                                   int64_t capacity, uint32_t* words, uint8_t* dts, int64_t* offsets, const emb_track_out* init,
                                   int64_t* total_rows) {
    return sample_events_impl(m, rng, n, T, opts, capacity, nullptr, words, dts, offsets, init, total_rows);
}

int64_t emb_model_get_gated(const emb_model* m, int32_t* buf, int64_t cap) {
    if (!m) return 0;
    const auto& g = m->h->gated;
    if (buf)
        for (size_t i = 0; i < g.size() && (int64_t)i < cap; ++i) buf[i] = g[i] + 1;
    return (int64_t)g.size();
}

int emb_dyn_limits_named(const char* ac_type, emb_dyn_limits* out) {
    if (!ac_type || !out) return set_err(EMB_E_ARG, "null argument");
    emb::TermLimits l;
    if (!emb::named_dyn_limits(ac_type, l)) return set_err(EMB_E_ARG, std::string("getDynamicLimits: unknown aircraft type ") + ac_type);
    *out = emb_dyn_limits{l.minVel, l.maxVel, l.maxTurn, l.maxAlt, l.maxVR};
    return 0;
}

int64_t emb_terminal_traj_len(int64_t n, double tmax_s) {
    if (n < 0 || !(tmax_s >= 0.0) || tmax_s >= 32767.0) return 0;
    return (int64_t)EMB_TRAJ_FIELDS * 2 * (2 * (int64_t)tmax_s + 1) * n;
}

int emb_terminal_propagate(const emb_terminal_models* models, const emb_rng* rng, int64_t n, const double* geo,
                           int64_t geo_stride, const int32_t* geo_rows, double tmax_s, const emb_dyn_limits* limits,
                           const emb_sample_opts* opts, const emb_traj_out* out) {
    if (!models || !rng || !geo_rows || !limits || !opts || !out || n < 0 || (n > 0 && !geo) || geo_stride < n)
        return set_err(EMB_E_ARG, "null or out-of-range argument");
    if (!(tmax_s >= 0.0) || tmax_s >= 32767.0) return set_err(EMB_E_ARG, "tmax_s must be in [0, 32767)");
    emb::TermParams P;
    std::memset(&P, 0, sizeof(P));
    P.seed = rng->seed;
    P.first_sample = rng->first_sample;
    P.n = n;
    P.tmax_s = tmax_s;
    emb::term_round_keys(P.seed, P.rk);
    P.tmax = (int32_t)tmax_s;
    P.max_attempts = opts->max_attempts > 0 ? std::min(opts->max_attempts, 65535) : 65535;
    P.geo_stride = geo_stride;
    int max_row = 0;
    for (int k = 0; k < 12; ++k) {
        if (geo_rows[k] < 0) return set_err(EMB_E_ARG, "geo_rows: negative row");
        P.geo_row[k] = geo_rows[k];
        max_row = std::max(max_row, (int)geo_rows[k]);
    }
    for (int a = 0; a < 2; ++a)
        P.lim[a] = emb::TermLimits{limits[a].minVel_ft_s, limits[a].maxVel_ft_s, limits[a].maxTurnRate_deg_s,
                                   limits[a].maxAltitude_ft, limits[a].maxVertRate_ft_s};
    constexpr size_t cuts_per_model = (size_t)emb::TERM_NCUT * emb::TERM_CUT_MAX;
    std::vector<double> cuts(cuts_per_model * emb::TERM_NMODELS);
    const emb_model* slot[emb::TERM_NMODELS] = {
        models->own_fwd[0], models->own_bck[0], models->own_fwd[1], models->own_bck[1], models->int_fwd[0],
        models->int_bck[0], models->int_fwd[1], models->int_bck[1], models->int_fwd[2], models->int_bck[2]};
    try {
        for (int k = 0; k < emb::TERM_NMODELS; ++k) {
            if (!slot[k]) return set_err(EMB_E_ARG, "emb_terminal_models: null model");
            emb::make_term_model(*slot[k]->h, P.lim[k < 4 ? 0 : 1], P.m[k], cuts.data() + (size_t)k * cuts_per_model);
        }
    } catch (const emb::Error& e) {
        return set_err(e.code, e.msg);
    }
    if (n == 0) return 0;
    int device, rc = 0;
    if ((rc = pick_device(opts, device))) return rc;
    for (int k = 0; k < emb::TERM_NMODELS; ++k) {
        DevModel D;
        if ((rc = ensure_device(*slot[k]->h, device, D))) return rc;
        P.m[k].thr = D.thr_trans;
        P.m[k].edges = D.edges;
    }
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    Stager sg{opts->mem, st, {}};
    struct Scratch {
        void* p = nullptr;
        ~Scratch() { tmp_free(p); }
    } d_geo, d_status, d_cuts;
    CU(tmp_alloc(&d_cuts.p, cuts.size() * 8, st));
    CU(cudaMemcpyAsync(d_cuts.p, cuts.data(), cuts.size() * 8, cudaMemcpyHostToDevice, st));   // pageable: staged before return
    P.cuts = (const double*)d_cuts.p;
    if (opts->mem == EMB_MEM_DEVICE) {
        P.geo = geo;
    } else {   // stage the rows that are read
        const size_t bytes = (size_t)(max_row + 1) * (size_t)geo_stride * 8;
        CU(tmp_alloc(&d_geo.p, bytes, st));
        CU(cudaMemcpyAsync(d_geo.p, geo, bytes, cudaMemcpyHostToDevice, st));
        P.geo = (const double*)d_geo.p;
    }
    emb::TermOut O{};
    if ((rc = sg.out(out->traj, (size_t)emb_terminal_traj_len(n, tmax_s) * 4, false, (void**)&O.traj))) return rc;
    if ((rc = sg.out(out->len, (size_t)n * 4 * 2, false, (void**)&O.len))) return rc;
    CU(tmp_alloc(&d_status.p, 4, st));
    CU(cudaMemsetAsync(d_status.p, 0, 4, st));
    O.status = (int32_t*)d_status.p;
    cudaError_t e = (cudaError_t)emb::launch_terminal(P, O, st);
    if (e != cudaSuccess) return cuda_fail(e, "launch k_terminal_chains");
    int32_t status = 0;
    CU(cudaMemcpyAsync(&status, d_status.p, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if ((rc = sg.finish())) return rc;
    if (status & 2) return set_err(EMB_E_ARG, "Unknown int_intent: own_intent must be 1..2 and int_intent 1..3 (createEncounter.m:22,37)");
    if (status & 1) return set_err(EMB_E_REJECT, "a trajectory state exhausted max_attempts in the dynamic-limit resample loop");
    return 0;
}

// ---- log-likelihood of given bins (emb_loglik.cuh) ------------------------------------------------------------------------
// the device status word of the scoring kernels -> EMB_E_ARG with what was wrong
static int loglik_status_error(int32_t status) {
    if (status & emb::LL_BAD_BIN) return set_err(EMB_E_ARG, "loglik: a bin is outside 1..r of its variable");
    if (status & emb::LL_BAD_COL0)
        return set_err(EMB_E_ARG, "loglik: column 0 of the track bins differs from init_bins of the dynamic variables");
    return 0;
}

// shared by both entry points: checks, device tables, staging, one launch, status
static int loglik_impl(const emb_model* m, int64_t n, int32_t T, const int8_t* init_bins, const int8_t* bins,
                       const emb_sample_opts* opts, double* initial, double* per_var, double* transition) {
    const bool tracks = T > 0;
    const HostModel& H = *m->h;
    if (opts->mem & ~0xFF) return set_err(EMB_E_ARG, "loglik: EMB_MEM_ASYNC is not supported; scoring calls are synchronous");
    if (n == 0) return 0;
    int device, rc = 0;
    if ((rc = pick_device(opts, device))) return rc;
    DevModel D;
    if ((rc = ensure_logp(H, device, D))) return rc;
    if (opts->correct_dbn) D.fast = 0;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    Stager sg{opts->mem, st, {}};
    const size_t ni = (size_t)H.n_initial;
    emb::LoglikParams P{};
    P.n = n;
    P.T = T;
    const void* d_in = nullptr;
    if ((rc = sg.in(init_bins, (size_t)n * ni, &d_in))) return rc;
    P.init_bins = (const int8_t*)d_in;
    if (tracks && (rc = sg.in(bins, (size_t)emb_tracks_bins_len(m, n, T), &d_in))) return rc;
    P.bins = tracks ? (const int8_t*)d_in : nullptr;
    if ((rc = sg.out(initial, (size_t)n * 8, false, (void**)&P.initial))) return rc;
    if ((rc = sg.out(per_var, (size_t)n * ni * 8, false, (void**)&P.per_var))) return rc;
    if ((rc = sg.out(transition, (size_t)n * 8, false, (void**)&P.transition))) return rc;
    CU(tmp_alloc((void**)&P.status, 4, st));
    CU(cudaMemsetAsync(P.status, 0, 4, st));
    cudaError_t e = tracks ? (cudaError_t)emb::launch_loglik_tracks(D, P, st)
                           : (cudaError_t)emb::launch_loglik_initial(D, P, (int)H.logp_initial.size(), st);
    if (e != cudaSuccess) {
        tmp_free(P.status);
        return cuda_fail(e, tracks ? "launch k_loglik_tracks" : "launch k_loglik_initial");
    }
    int32_t status = 0;
    e = cudaMemcpyAsync(&status, P.status, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    tmp_free(P.status);
    if (e != cudaSuccess) return cuda_fail(e, tracks ? "k_loglik_tracks" : "k_loglik_initial");
    if ((rc = sg.finish())) return rc;
    return loglik_status_error(status);
}

int emb_loglik_initial(const emb_model* m, int64_t n, const int8_t* bins, const emb_sample_opts* opts, double* total,
                       double* per_var) {
    if (!m || !opts || n < 0 || (n > 0 && (!bins || !total))) return set_err(EMB_E_ARG, "null or out-of-range argument");
    return loglik_impl(m, n, 0, bins, nullptr, opts, total, per_var, nullptr);
}

int emb_loglik_tracks(const emb_model* m, int64_t n, int32_t T, const int8_t* init_bins, const int8_t* bins,
                      const emb_sample_opts* opts, double* initial, double* transition) {
    if (!m || !opts || n < 0 || T < 1 || (n > 0 && (!init_bins || !bins)))
        return set_err(EMB_E_ARG, "null or out-of-range argument");
    const HostModel& H = *m->h;
    if (!H.has_transition || H.temporal_map.empty())
        return set_err(EMB_E_ARG, "dynvar:empty: model has no transition network");
    return loglik_impl(m, n, T, init_bins, bins, opts, initial, nullptr, transition);
}

// IntegrateParams from emb_integrate_opts (labels -> tile ordinals, unit ratios); 0 or an error code
static int fill_integrate(const HostModel& H, const emb_integrate_opts* opts, int64_t n, int32_t T, emb::IntegrateParams& P) {
    std::memset(&P, 0, sizeof(P));
    P.n = n;
    P.T = T;
    auto tv_of = [&](int32_t var1) -> int {
        for (size_t k = 0; k < H.timevarying.size(); ++k)
            if (H.timevarying[k] == var1 - 1) return (int)k;
        return -1;
    };
    if (opts->idx_altitude < 1 || opts->idx_altitude > H.n_initial || opts->idx_speed < 1 || opts->idx_speed > H.n_initial)
        return set_err(EMB_E_ARG, "sample2track: idx_altitude / idx_speed must name initial variables");
    P.i_alt = opts->idx_altitude - 1;
    P.i_speed = opts->idx_speed - 1;
    P.g_acc = tv_of(opts->idx_acceleration);
    P.g_vr = tv_of(opts->idx_vertrate);
    P.g_turn = tv_of(opts->idx_turnrate);
    P.n_tv = (int32_t)H.timevarying.size();
    if (P.g_acc < 0 || P.g_vr < 0 || P.g_turn < 0)
        return set_err(EMB_E_ARG, "sample2track: acceleration, vertical rate and turn rate must be time-varying variables of the model");
    P.ur_speed = opts->ur_speed;
    P.ur_vertrate = opts->ur_vertrate;
    P.ur_heading = opts->ur_heading;
    P.min_speed = opts->min_speed;
    P.max_speed = opts->max_speed;
    return 0;
}

int emb_tracks_integrate(const emb_model* m, int64_t n, int32_t T, const double* init_values, const float* values,
                         const emb_integrate_opts* opts, float* xyz, uint8_t* is_good) {
    if (!m || !opts || n < 0 || T < 1 || (n > 0 && (!init_values || !values)))
        return set_err(EMB_E_ARG, "null or out-of-range argument");
    const HostModel& H = *m->h;
    emb::IntegrateParams P;
    if (int rcf = fill_integrate(H, opts, n, T, P)) return rcf;
    if (n == 0) return 0;
    emb_sample_opts so;
    emb_sample_opts_init(&so);
    so.device = opts->device;
    int device, rc = 0;
    if ((rc = pick_device(&so, device))) return rc;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    Stager sg{opts->mem, st, {}};
    struct Scratch {
        void* p = nullptr;
        ~Scratch() { tmp_free(p); }
    } d_init, d_vals;
    const size_t init_bytes = (size_t)H.n_initial * (size_t)n * 8;
    const size_t val_bytes = (size_t)emb_tracks_values_len(m, n, T) * 4;
    if (opts->mem == EMB_MEM_DEVICE) {
        P.init_values = init_values;
        P.values = values;
    } else {
        CU(tmp_alloc(&d_init.p, init_bytes, st));
        CU(tmp_alloc(&d_vals.p, val_bytes, st));
        CU(cudaMemcpyAsync(d_init.p, init_values, init_bytes, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_vals.p, values, val_bytes, cudaMemcpyHostToDevice, st));
        P.init_values = (const double*)d_init.p;
        P.values = (const float*)d_vals.p;
    }
    if ((rc = sg.out(xyz, (size_t)3 * (size_t)(T + 1) * (size_t)n * 4, false, (void**)&P.xyz))) return rc;
    if ((rc = sg.out(is_good, (size_t)n, false, (void**)&P.is_good))) return rc;
    cudaError_t e = (cudaError_t)emb::launch_integrate(P, st);
    if (e != cudaSuccess) return cuda_fail(e, "launch k_tracks_integrate");
    CU(cudaStreamSynchronize(st));
    return sg.finish();
}

int emb_sample_tracks_xyz(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                          const emb_integrate_opts* iopts, const emb_track_out* out, float* xyz, uint8_t* is_good) {
    if (!m || !rng || !opts || !iopts || n < 0 || T < 1) return set_err(EMB_E_ARG, "null or out-of-range argument");
    if (out && (out->hist_initial || out->hist_transition))
        return set_err(EMB_E_ARG, "emb_sample_tracks_xyz: histograms belong to emb_sample_tracks");
    if (opts->mem & EMB_MEM_ASYNC) return set_err(EMB_E_ARG, "emb_sample_tracks_xyz: EMB_MEM_ASYNC is not supported");
    const HostModel& H = *m->h;
    if (!H.has_transition || H.temporal_map.empty())
        return set_err(EMB_E_ARG, "dynvar:empty: model has no transition network");
    if ((int64_t)T * (int64_t)H.gated.size() >= (1ll << 33))
        return set_err(EMB_E_LIMIT, "T too large for the 32-bit stream index");
    emb::SampleParams P;
    emb::IntegrateParams IP;
    int rc = 0;
    try {
        emb::fill_params(H, rng->seed, rng->first_sample, n, T, *opts, P);
    } catch (const emb::Error& e) {
        return set_err(e.code, e.msg);
    }
    if ((rc = fill_integrate(H, iopts, n, T, IP))) return rc;
    if (n == 0) return 0;
    int device;
    if ((rc = pick_device(opts, device, true))) return rc;
    DevModel D;
    if ((rc = ensure_device(H, device, D))) return rc;
    if (opts->correct_dbn) D.fast = 0;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    Stager sg{opts->mem & 0xFF, st, {}};
    emb::TrackOut O{};
    const size_t ni = (size_t)H.n_initial;
    const emb_track_out none{};
    const emb_track_out* o = out ? out : &none;
    if ((rc = sg.out(o->bins, (size_t)emb_tracks_bins_len(m, n, T), false, (void**)&O.bins))) return rc;
    if ((rc = sg.out(o->values, (size_t)emb_tracks_values_len(m, n, T) * 4, false, (void**)&O.values))) return rc;
    if ((rc = sg.out(o->init_bins, (size_t)n * ni, false, (void**)&O.init_bins))) return rc;
    if ((rc = sg.out(o->init_values, (size_t)n * ni * 8, false, (void**)&O.init_values))) return rc;
    if ((rc = sg.out(o->attempts, (size_t)n * 2, false, (void**)&O.attempts))) return rc;
    if ((rc = sg.out(xyz, (size_t)3 * (size_t)(T + 1) * (size_t)n * 4, false, (void**)&O.x.xyz))) return rc;
    if ((rc = sg.out(is_good, (size_t)n, false, (void**)&O.x.is_good))) return rc;
    if (!O.x.xyz && !O.x.is_good) return set_err(EMB_E_ARG, "emb_sample_tracks_xyz: xyz and is_good are both null");
    O.x.g_acc = IP.g_acc; O.x.g_vr = IP.g_vr; O.x.g_turn = IP.g_turn; O.x.i_alt = IP.i_alt; O.x.i_speed = IP.i_speed;
    O.x.ur_speed = IP.ur_speed; O.x.ur_vertrate = IP.ur_vertrate; O.x.ur_heading = IP.ur_heading;
    O.x.min_speed = IP.min_speed; O.x.max_speed = IP.max_speed;
    if ((rc = stage_start(sg, opts, H, n, P))) return rc;
    struct Scratch {
        void* p = nullptr;
        ~Scratch() { tmp_free(p); }
    } d_status, d_values, d_inits;
    CU(tmp_alloc(&d_status.p, 4, st));
    CU(cudaMemsetAsync(d_status.p, 0, 4, st));
    O.status = (int32_t*)d_status.p;
    int le = emb::launch_tracks(D, P, O, st);
    if (le == -1) {   // no fused kernel for this shape: sample the dense values (into a temporary if the caller wants none), then integrate
        emb::TrackOut O2 = O;
        O2.x = emb::XyzOut{};
        if (!O2.values) {
            CU(tmp_alloc(&d_values.p, (size_t)emb_tracks_values_len(m, n, T) * 4, st));
            O2.values = (float*)d_values.p;
        }
        if (!O2.init_values) {
            CU(tmp_alloc(&d_inits.p, (size_t)n * ni * 8, st));
            O2.init_values = (double*)d_inits.p;
        }
        le = emb::launch_tracks(D, P, O2, st);
        if (le == 0) {
            IP.init_values = O2.init_values;
            IP.values = O2.values;
            IP.xyz = O.x.xyz;
            IP.is_good = O.x.is_good;
            le = emb::launch_integrate(IP, st);
        }
    }
    if (le != 0) return cuda_fail((cudaError_t)le, "launch k_tracks (xyz)");
    int32_t status = 0;
    CU(cudaMemcpyAsync(&status, d_status.p, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if ((rc = sg.finish())) return rc;
    return status_error(status);
}

int emb_terminal_screen(const float* traj, const int16_t* len, int64_t n, double tmax_s, double thres_dist_ft,
                        double thres_altlow_ft, const emb_sample_opts* opts, const emb_screen_out* out) {
    if (!opts || !out || n < 0 || (n > 0 && (!traj || !len))) return set_err(EMB_E_ARG, "null or out-of-range argument");
    if (!(tmax_s >= 0.0) || tmax_s >= 32767.0) return set_err(EMB_E_ARG, "tmax_s must be in [0, 32767)");
    if (n == 0) return 0;
    int device, rc = 0;
    if ((rc = pick_device(opts, device))) return rc;
    cudaStream_t st = (cudaStream_t)opts->stream;
    g_call_stream = st;
    emb::ScreenParams P;
    std::memset(&P, 0, sizeof(P));
    P.n = n;
    P.tmax = (int32_t)tmax_s;
    P.thres_dist_ft = thres_dist_ft;
    P.thres_altlow_ft = thres_altlow_ft;
    struct Scratch {
        void* p = nullptr;
        ~Scratch() { tmp_free(p); }
    } d_traj, d_len;
    const size_t tb = (size_t)emb_terminal_traj_len(n, tmax_s) * 4, lb = (size_t)n * 4 * 2;
    if (opts->mem == EMB_MEM_DEVICE) {
        P.traj = traj;
        P.len = len;
    } else {
        CU(tmp_alloc(&d_traj.p, tb, st));
        CU(tmp_alloc(&d_len.p, lb, st));
        CU(cudaMemcpyAsync(d_traj.p, traj, tb, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_len.p, len, lb, cudaMemcpyHostToDevice, st));
        P.traj = (const float*)d_traj.p;
        P.len = (const int16_t*)d_len.p;
    }
    Stager sg{opts->mem, st, {}};
    if ((rc = sg.out(out->hmd_ft, (size_t)n * 8, false, (void**)&P.hmd_ft))) return rc;
    if ((rc = sg.out(out->vmd_ft, (size_t)n * 8, false, (void**)&P.vmd_ft))) return rc;
    if ((rc = sg.out(out->tcpa, (size_t)n * 3 * 2, false, (void**)&P.tcpa))) return rc;
    if ((rc = sg.out(out->enc_time_s, (size_t)n * 2, false, (void**)&P.enc_time_s))) return rc;
    if ((rc = sg.out(out->runway, (size_t)n, false, (void**)&P.runway))) return rc;
    cudaError_t e = (cudaError_t)emb::launch_screen(P, st);
    if (e != cudaSuccess) return cuda_fail(e, "launch k_terminal_screen");
    CU(cudaStreamSynchronize(st));
    return sg.finish();
}

}  // extern "C"
