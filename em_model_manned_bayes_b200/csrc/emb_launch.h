// emb_launch.h -- launchers implemented in emb_kernels.cu, called from the C-ABI layer.
#pragma once
#include <atomic>
#include <cstdint>

#include "emb_device.cuh"

namespace emb {

extern std::atomic<long long> g_launch_count;
extern std::atomic<int> g_force_generic;
extern std::atomic<int> g_last_kernel_fast;

// all return a cudaError_t value (0 = success); pointers are device pointers
// table_words = length of the initial threshold table (decides shared-memory staging)
int launch_initial(const DevModel& M, const SampleParams& P, int table_words, int8_t* bins, double* values,
                   uint16_t* attempts, unsigned long long* hist, int32_t* status, void* stream);
int launch_initial_f32(const DevModel& M, const SampleParams& P, int table_words, int8_t* bins, float* values,
                       uint16_t* attempts, unsigned long long* hist, int32_t* status, void* stream);
int launch_tracks(const DevModel& M, const SampleParams& P, const TrackOut& O, void* stream);
// offsets[0..n] = carry + exclusive prefix sums of counts[0..n), offsets[n] = carry + total; carry = *carry_in (device pointer,
// may alias offsets) or 0; scratch: scan_scratch_len(n) long longs
long long scan_scratch_len(long long n);
int launch_scan_counts(const uint32_t* counts, long long* offsets, long long n, long long* scratch, void* stream,
                       const long long* carry_in = nullptr);

// packed event rows [first, first + count) (emb_device.cuh: pack_event_word) -> 8-byte emb_event rows at the same indices
int launch_expand_events(const DevModel& M, const uint32_t* words, const uint8_t* dts, void* rows, long long first, long long count,
                         const EventFormat& fm, void* stream);

// {*total, *flag} written by an SM into mapped pinned host memory (two long longs)
int launch_publish(const long long* total, const int32_t* flag, long long* mapped_dst, void* stream);

// log-likelihood of given bins (emb_loglik.cuh); M.logp_init / M.logp_trans set; table_len = slots of the initial table
struct LoglikParams;
int launch_loglik_initial(const DevModel& M, const LoglikParams& P, int table_len, void* stream);
// M.fast selects the branch: frozen parents (counting kernel) or per-step parents
int launch_loglik_tracks(const DevModel& M, const LoglikParams& P, void* stream);

// terminal trajectory chains (emb_terminal.cu): 4 chains per encounter
struct TermParams;
struct TermOut;
int launch_terminal(const TermParams& P, const TermOut& O, void* stream);

struct ScreenParams;
int launch_screen(const ScreenParams& P, void* stream);
// first-order track integration (sample2track.m Euler loop) over the dense tiles
struct IntegrateParams;
int launch_integrate(const IntegrateParams& P, void* stream);

}  // namespace emb
