// emb_kernels.cu -- sm_100a kernels of libemb200.so and their launchers.
//
// One thread = one sample (track).  There is no inter-thread communication on the data path; the
// only shared state is the per-block verification histogram (shared-memory atomics flushed with one
// global atomic per bin per block).
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>

#include "emb_device.cuh"
#include "emb_events_expand.cuh"
#include "emb_fast.cuh"
#include "emb_format.cuh"
#include "emb_initial.cuh"
#include "emb_launch.h"
#include "emb_loglik.cuh"
#include "emb_loglik_events.cuh"
#include "emb_parse.cuh"

namespace emb {

std::atomic<long long> g_launch_count{0};
std::atomic<int> g_force_generic{0};      // emb_debug_force_generic(): tests compare both kernels
std::atomic<int> g_last_kernel_fast{0};

namespace {

#ifndef EMB_BLOCK
#define EMB_BLOCK 128
#endif
#ifndef EMB_MINBLOCKS
#define EMB_MINBLOCKS 4
#endif
#ifndef EMB_MINBLOCKS_XYZ       // fused integration (mode 3): five more fp64 state words and a sincosd per second
#define EMB_MINBLOCKS_XYZ 4
#endif
#ifndef EMB_MINBLOCKS_SLOW      // slow branch (per-second column gathers): latency-bound, more resident warps help -- as long as
#define EMB_MINBLOCKS_SLOW 5    // the columns of all dynamic variables still fit in registers (four 9-bin variables need 128)
#endif
constexpr int BLOCK = EMB_BLOCK;

struct SmemHist {
    uint32_t* sh;
    __device__ __forceinline__ void operator()(int which, int idx, int bin) const {
        atomicAdd(&sh[(which ? MAXV * HIST_STRIDE : 0) + idx * HIST_STRIDE + bin], 1u);
    }
};

__device__ __forceinline__ void flush_hist(const uint32_t* sh, const DevModel& M, unsigned long long* hi,
                                           unsigned long long* ht) {
    __syncthreads();
    if (hi)
        for (int q = threadIdx.x; q < M.n_initial * HIST_STRIDE; q += blockDim.x)
            if (sh[q]) atomicAdd(&hi[q], (unsigned long long)sh[q]);
    if (ht)
        for (int q = threadIdx.x; q < M.n_dyn * HIST_STRIDE; q += blockDim.x)
            if (sh[MAXV * HIST_STRIDE + q]) atomicAdd(&ht[q], (unsigned long long)sh[MAXV * HIST_STRIDE + q]);
}

// ---- initial network only (bn_sample.m batch; config 2; terminal geometry) ----------------------
template <class VT>
__global__ void __launch_bounds__(BLOCK)
k_initial(const __grid_constant__ DevModel M, const __grid_constant__ SampleParams P, int8_t* __restrict__ bins,
          VT* __restrict__ values, uint16_t* __restrict__ attempts, unsigned long long* hist, int32_t* status) {
    __shared__ uint32_t sh[MAXV * HIST_STRIDE];
    if (hist) {
        for (int q = threadIdx.x; q < MAXV * HIST_STRIDE; q += blockDim.x) sh[q] = 0;
        __syncthreads();
    }
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < P.n) {
        uint8_t x[MAXX];
        double vals[MAXV];
        int attempt = sample_initial(M, P, P.first_sample + (uint64_t)s, x, vals);
        if (attempt < 0) {
            *status = attempt == -2 ? 2 : 1;
            attempt = P.max_attempts;
        }
        if (attempts) attempts[s] = (uint16_t)(attempt + 1);
        for (int i = 0; i < M.n_initial; ++i) {
            if (bins) bins[(int64_t)i * P.n + s] = (int8_t)(x[i] + 1);
            if (values) values[(int64_t)i * P.n + s] = (VT)vals[i];
            if (hist) atomicAdd(&sh[i * HIST_STRIDE + x[i]], 1u);
        }
    }
    if (hist) flush_hist(sh, M, hist, nullptr);
}

// ---- initial network, register-resident (emb_initial.cuh): 4 consecutive samples per thread -------
// SMEM: the whole threshold table (glider family 42 KB, balloons, HAA transition-free models ...) is
// staged in shared memory once per persistent block, so the per-lane column gathers are LDS.128
// instead of 32-sector L1 lookups; larger tables (7-variable uncor: 0.6-1.1 MB) are gathered from L1/L2.
#ifndef EMB_INIT_MINBLOCKS_V    // resident blocks asked of the values variant (its fp64 tail otherwise takes 102 registers)
#define EMB_INIT_MINBLOCKS_V 3
#endif
#ifndef EMB_INIT_TMA            // 1: stage the threshold table with TMA bulk copies (unpadded); 0: __ldg loop into the padded layout
#define EMB_INIT_TMA 0
#endif
#ifndef EMB_INIT_PAD            // words between consecutive columns of the shared-memory copy (0 with EMB_INIT_TMA)
#define EMB_INIT_PAD (EMB_INIT_TMA ? 0 : 4)
#endif
#ifndef EMB_INIT_MINBLOCKS_B
#define EMB_INIT_MINBLOCKS_B 3
#endif
template <int NV, bool VALUES, bool SMEM, class VT, bool ALIGNED>
__global__ void __launch_bounds__(256, VALUES ? EMB_INIT_MINBLOCKS_V : EMB_INIT_MINBLOCKS_B)
k_initial_fast(const __grid_constant__ DevModel M, const __grid_constant__ SampleParams P,
               const __grid_constant__ InitStrides ST, const __grid_constant__ InitCalls IC, int table_words,
               int8_t* __restrict__ bins, VT* __restrict__ values, uint16_t* __restrict__ attempts) {
    extern __shared__ uint4 smem_table[];
    const uint32_t* table = M.thr_init;
    if (SMEM) {
#if EMB_INIT_TMA
        // A/B variant (profiles/r2_init_staging_tma_vs_ldg.txt): the table as ONE linear image, moved by the TMA unit with
        // 1-D bulk copies (cp.async.bulk, SASS UBLKCP) that complete on an mbarrier -- requires the unpadded layout
        // (ST.pad == 0: the bulk copy cannot re-pitch columns), which costs more in LDS bank conflicts than the copy saves.
        __shared__ __align__(8) unsigned long long mbar;
        const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&mbar);
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_table);
        const uint32_t bytes = (uint32_t)table_words * 4u;
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
            for (uint32_t o = 0; o < bytes; o += 16384u) {
                const uint32_t len = bytes - o < 16384u ? bytes - o : 16384u;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst + o), "l"(reinterpret_cast<const char*>(M.thr_init) + o), "r"(len), "r"(mb) : "memory");
            }
        }
        __syncthreads();
        {
            uint32_t done = 0;
            while (!done)
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(done) : "r"(mb) : "memory");
        }
#else
        // copy with a pitch of rp + pad words per column (emb_initial.cuh: fill_init_strides)
        const uint4* src = reinterpret_cast<const uint4*>(M.thr_init);
        for (int q = threadIdx.x; q < table_words / 4; q += blockDim.x) {
            const uint32_t w = 4u * (uint32_t)q;
            int i = 0;
#pragma unroll
            for (int v = 1; v < NV; ++v) i += w >= ST.src_off[v] ? 1 : 0;
            const uint32_t rel = w - ST.src_off[i], c = rel / ST.rp[i], r = rel - c * ST.rp[i];
            smem_table[(ST.off[i] + c * (ST.rp[i] + ST.pad) + r) / 4] = __ldg(src + q);
        }
        __syncthreads();
#endif
        table = reinterpret_cast<const uint32_t*>(smem_table);
    }
    // fp32 de-discretisation entries of the initial variables (16 bytes per bin): shared memory as well
    __shared__ float4 s_ent[VALUES && sizeof(VT) == 4 ? 256 : 1];
    const float* ent = M.dd32 + 4 * M.ddi_off[0];
    if (VALUES && sizeof(VT) == 4) {
        int total = 0;
#pragma unroll
        for (int v = 0; v < NV; ++v) total += M.init[v].r;
        if (total <= 256) {
            for (int q = threadIdx.x; q < total; q += blockDim.x) s_ent[q] = __ldg(reinterpret_cast<const float4*>(ent) + q);
            ent = reinterpret_cast<const float*>(s_ent);
        }
    }
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * INIT_SPT;
    for (int64_t s0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * INIT_SPT; s0 < P.n; s0 += stride)
        initial_fast4<NV, VALUES, VT, ALIGNED>(M, P, ST, IC, table, ent, s0, bins, values, attempts);
}

// ---- tracks, generic (any model, both dbn_sample.m branches) ------------------------------------
__global__ void __launch_bounds__(BLOCK)
k_tracks_generic(const __grid_constant__ DevModel M, const __grid_constant__ SampleParams P,
                 const __grid_constant__ TrackOut O) {
    __shared__ uint32_t sh[(MAXV + MAXD) * HIST_STRIDE];
    const bool want_hist = O.hist_initial || O.hist_transition;
    if (want_hist) {
        for (int q = threadIdx.x; q < (MAXV + MAXD) * HIST_STRIDE; q += blockDim.x) sh[q] = 0;
        __syncthreads();
    }
    const int64_t s = P.s_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < P.s_end) track_generic(M, P, O, s, SmemHist{sh});
    else if (P.s_end == P.n) zero_padding_track(O, M.n_dyn, M.n_gated, P.T, P.n, s);
    if (want_hist) flush_hist(sh, M, O.hist_initial, O.hist_transition);
}

// ---- tracks, register-resident specialisation (emb_fast.cuh) --------------------------------------
template <uint32_t RS, int NG, bool FAST, bool HIST, int EV, uint32_t ORD>
__global__ void __launch_bounds__(BLOCK, EV == 3 ? EMB_MINBLOCKS_XYZ : FAST ? EMB_MINBLOCKS : (DynShape<RS>::ND >= 4 ? EMB_MINBLOCKS : EMB_MINBLOCKS_SLOW))
k_tracks_fast(const __grid_constant__ DevModel M, const __grid_constant__ SampleParams P,
              const __grid_constant__ TrackOut O) {
    __shared__ FastShared S;
    __shared__ CallTable<NG> U;
    __shared__ uint32_t sh[HIST ? (MAXV + MAXD) * HIST_STRIDE : 1];
    fast_fill_shared(M, S, threadIdx.x, blockDim.x);
    if (HIST)
        for (int q = threadIdx.x; q < (MAXV + MAXD) * HIST_STRIDE; q += blockDim.x) sh[q] = 0;
    __syncthreads();
    const int64_t s = P.s_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    track_fast<RS, NG, FAST, HIST, EV, ORD>(M, P, O, s, s < P.s_end, S, U, (int)threadIdx.x, (int)blockDim.x, SmemHist{sh});
    if (!ev_list(EV) && s >= P.s_end && P.s_end == P.n) zero_padding_track(O, M.n_dyn, NG, P.T, P.n, s);
    if (HIST) flush_hist(sh, M, O.hist_initial, O.hist_transition);
}

// ---- exclusive prefix sum of the per-track row counts: tile sums, scan of the tile sums, tile-local scans ------
constexpr int SCAN_THREADS = 256, SCAN_PER_THREAD = 8, SCAN_TILE = SCAN_THREADS * SCAN_PER_THREAD;

__device__ __forceinline__ long long block_exclusive_scan(long long v, long long* warp_sum, long long* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[w] = x;
    __syncthreads();
    if (w == 0) {
        long long t = lane < nw ? warp_sum[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xFFFFFFFFu, t, o);
            if (lane >= o) t += y;
        }
        warp_sum[lane] = t;
    }
    __syncthreads();
    const long long before = (w ? warp_sum[w - 1] : 0) + x - v;
    if (total) *total = warp_sum[nw - 1];
    __syncthreads();
    return before;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_sums(const uint32_t* __restrict__ counts, long long* __restrict__ tile_sum,
                                                                 long long n) {
    __shared__ long long warp_sum[32];
    const long long base = (long long)blockIdx.x * SCAN_TILE + (long long)threadIdx.x * SCAN_PER_THREAD;
    long long v = 0;
#pragma unroll
    for (int q = 0; q < SCAN_PER_THREAD; ++q)
        if (base + q < n) v += counts[base + q];
    long long total;
    block_exclusive_scan(v, warp_sum, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// one block: tile_sum[0..m) -> exclusive prefixes in place, grand total to *total_out
// carry_in (nullable): value the prefixes start from (the total of the tracks before this range)
__global__ void __launch_bounds__(1024) k_scan_tile_prefix(long long* __restrict__ tile_sum, long long m, long long* __restrict__ total_out,
                                                           const long long* __restrict__ carry_in) {
    __shared__ long long warp_sum[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = carry_in ? *carry_in : 0;
    __syncthreads();
    for (long long base = 0; base < m; base += 1024) {
        const long long i = base + threadIdx.x;
        const long long v = i < m ? tile_sum[i] : 0;
        long long total;
        const long long before = block_exclusive_scan(v, warp_sum, &total);
        if (i < m) tile_sum[i] = carry + before;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(const uint32_t* __restrict__ counts, const long long* __restrict__ tile_prefix,
                                                             long long* __restrict__ offsets, long long n) {
    __shared__ long long warp_sum[32];
    const long long base = (long long)blockIdx.x * SCAN_TILE + (long long)threadIdx.x * SCAN_PER_THREAD;
    uint32_t c[SCAN_PER_THREAD];
    long long v = 0;
#pragma unroll
    for (int q = 0; q < SCAN_PER_THREAD; ++q) {
        c[q] = base + q < n ? counts[base + q] : 0u;
        v += c[q];
    }
    long long run = tile_prefix[blockIdx.x] + block_exclusive_scan(v, warp_sum, nullptr);
#pragma unroll
    for (int q = 0; q < SCAN_PER_THREAD; ++q) {
        if (base + q < n) offsets[base + q] = run;
        run += c[q];
    }
}

// packed rows [first, first + count) -> 8-byte emb_event rows (emb_device.cuh: expand_event)
__global__ void __launch_bounds__(256) k_expand_events(const __grid_constant__ DevModel M, const uint32_t* __restrict__ words,
                                                       const uint8_t* __restrict__ dts, uint2* __restrict__ rows,
                                                       long long first, long long count, EventFormat fm) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t dt_lo = fm.dt_bytes == 1 ? (uint32_t)__ldg(dts + first + i)
                                            : (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(dts) + first + i);
    rows[first + i] = expand_event(M, __ldg(words + first + i), dt_lo, fm);
}

// {*total, *flag} -> dst (mapped host memory): a store from an SM does not queue behind the row copies on the copy engine,
// which a cudaMemcpy of the same eight bytes would
__global__ void k_publish(const long long* __restrict__ total, const int32_t* __restrict__ flag, volatile long long* dst) {
    dst[0] = *total;
    dst[1] = (long long)*flag;
}


// ---- log-likelihood of given bins (emb_loglik.cuh) -----------------------------------------------------------------------
// initial network: one thread per sample, grid-stride over a persistent grid; with SMEM the whole fp64 table is staged in shared
// memory once per block (glider: 9 156 slots, 73 KB), so the per-variable gathers are LDS instead of L1/L2 lookups
template <bool SMEM>
__global__ void __launch_bounds__(256) k_loglik_initial(const __grid_constant__ DevModel M, const __grid_constant__ LoglikParams P,
                                                        int table_len) {
    extern __shared__ double s_logp[];
    const double* logp = M.logp_init;
    if (SMEM) {
        for (int q = threadIdx.x; q < table_len; q += blockDim.x) s_logp[q] = __ldg(M.logp_init + q);
        __syncthreads();
        logp = s_logp;
    }
    uint8_t x[MAXV];
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < P.n; s += (int64_t)gridDim.x * blockDim.x) {
        const double v = loglik_initial_one(M, logp, P, s, x);
        if (P.initial) P.initial[s] = v;
    }
}

// tracks: one thread per track.  FROZEN: per-thread counters in dynamic shared memory laid out [counter][thread] (consecutive
// threads in consecutive banks), one byte extract + shared increment per variable-second; otherwise per-second gathers.
template <bool FROZEN>
__global__ void __launch_bounds__(128) k_loglik_tracks(const __grid_constant__ DevModel M, const __grid_constant__ LoglikParams P) {
    extern __shared__ uint32_t s_cnt[];
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= P.n) return;
    const int tid = threadIdx.x, bs = blockDim.x;
    loglik_track(M, P, s, FROZEN, [&](int k) -> uint32_t& { return s_cnt[k * bs + tid]; });
}

// tracks as event lists: one thread per track walking its rows, the dynamic state in a register; FROZEN counters as k_loglik_tracks
template <bool PACKED, bool FROZEN>
__global__ void __launch_bounds__(128) k_loglik_events(const __grid_constant__ DevModel M, const __grid_constant__ LoglikParams P,
                                                       const __grid_constant__ EventRows R) {
    extern __shared__ uint32_t s_cnt[];
    __shared__ int8_t s_dyn[MAXV];
    if (threadIdx.x < MAXV) s_dyn[threadIdx.x] = (int8_t)ll_dyn_of(M, threadIdx.x);
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= P.n) return;
    const int tid = threadIdx.x, bs = blockDim.x;
    loglik_track_events<PACKED>(M, P, R, s_dyn, s, FROZEN, [&](int k) -> uint32_t& { return s_cnt[k * bs + tid]; });
}

// event lists -> samples and control rows (emb_events_expand.cuh): one warp per track
constexpr int EE_BLOCK = 256;

template <bool PACKED>
__global__ void __launch_bounds__(EE_BLOCK) k_events_expand_count(const __grid_constant__ DevModel M,
                                                                  const __grid_constant__ ExpandParams P,
                                                                  const __grid_constant__ EventRows R) {
    const int64_t s = (int64_t)blockIdx.x * (EE_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    const ExpandLanes L{(int)(threadIdx.x & 31)};
    const uint32_t rows = events_expand_count<PACKED>(M, P, R, s, L);
    if (L.lane == 0) P.counts[s] = rows;
}

template <bool PACKED>
__global__ void __launch_bounds__(EE_BLOCK) k_events_expand(const __grid_constant__ DevModel M, const __grid_constant__ ExpandParams P,
                                                            const __grid_constant__ EventRows R) {
    __shared__ ExpandShared sh[EE_BLOCK / 32];
    const int64_t s = (int64_t)blockIdx.x * (EE_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    events_expand_track<PACKED>(M, P, R, s, ExpandLanes{(int)(threadIdx.x & 31)}, sh[threadIdx.x >> 5]);
}

// the text files of em_sample.m (emb_format.cuh): one warp per track, count pass and write pass of each file.  128 registers
// (16 warps an SM) hold the digit generation without spills; the default heuristic spills it.
constexpr int FMT_BLOCK = 128;
constexpr int FMT_MAXNREG = 128;

template <bool TRANS>
__device__ __forceinline__ void format_count(const FormatParams& P) {
    const int64_t s = (int64_t)blockIdx.x * (FMT_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    const ExpandLanes L{(int)(threadIdx.x & 31)};
    const uint32_t bytes = format_track<TRANS, false>(P, s, L, nullptr);
    if (L.lane == 0) P.counts[s] = bytes;
}
template <bool TRANS>
__device__ __forceinline__ void format_write(const FormatParams& P) {
    __shared__ char stage[FMT_BLOCK / 32][FMT_STAGE_BYTES];
    const int64_t s = (int64_t)blockIdx.x * (FMT_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    format_track<TRANS, true>(P, s, ExpandLanes{(int)(threadIdx.x & 31)}, stage[threadIdx.x >> 5]);
}
__global__ void __maxnreg__(FMT_MAXNREG) k_format_initial_count(const __grid_constant__ FormatParams P) { format_count<false>(P); }
__global__ void __maxnreg__(FMT_MAXNREG) k_format_initial(const __grid_constant__ FormatParams P) { format_write<false>(P); }
__global__ void __maxnreg__(FMT_MAXNREG) k_format_transition_count(const __grid_constant__ FormatParams P) { format_count<true>(P); }
__global__ void __maxnreg__(FMT_MAXNREG) k_format_transition(const __grid_constant__ FormatParams P) { format_write<true>(P); }

// the CSV rows of sample2track.m (emb_format.cuh: format_csv_track), the same shape and register cap
__global__ void __maxnreg__(FMT_MAXNREG) k_format_csv_count(const __grid_constant__ CsvParams P) {
    const int64_t s = (int64_t)blockIdx.x * (FMT_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    const ExpandLanes L{(int)(threadIdx.x & 31)};
    const uint32_t bytes = format_csv_track<false>(P, s, L, nullptr);
    if (L.lane == 0) P.counts[s] = bytes;
}
__global__ void __maxnreg__(FMT_MAXNREG) k_format_csv(const __grid_constant__ CsvParams P) {
    __shared__ char stage[FMT_BLOCK / 32][FMT_STAGE_BYTES];
    const int64_t s = (int64_t)blockIdx.x * (FMT_BLOCK / 32) + (threadIdx.x >> 5);
    if (s >= P.n) return;
    format_csv_track<true>(P, s, ExpandLanes{(int)(threadIdx.x & 31)}, stage[threadIdx.x >> 5]);
}

// decimal text tables (emb_parse.cuh).  Line discovery: one warp per PARSE_CHUNK bytes, each lane 16 bytes per round (one vector
// load when the text is 16-byte aligned); then one thread per line for the checks and for the values.
constexpr int PARSE_BLOCK = 256;
constexpr int PARSE_CHUNK = 4096;
constexpr int PARSE_ROUNDS = PARSE_CHUNK / 512;

// the 16 bytes at pos, zeros past the end of the text
__device__ __forceinline__ uint4 parse_load16(const ParseParams& P, int64_t pos) {
    if (P.aligned && pos + 16 <= P.bytes) return __ldg(reinterpret_cast<const uint4*>(P.text + pos));
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int b = 0; b < 16; ++b)
        if (pos + b < P.bytes) w[b >> 2] |= (uint32_t)(uint8_t)P.text[pos + b] << (8 * (b & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ uint32_t parse_nl4(uint32_t x) { return __vcmpeq4(x, 0x0A0A0A0Au); }   // 0xFF in each '\n' byte
__device__ __forceinline__ int parse_nl16(const uint4& v) {
    return (__popc(parse_nl4(v.x)) + __popc(parse_nl4(v.y)) + __popc(parse_nl4(v.z)) + __popc(parse_nl4(v.w))) >> 3;
}

__global__ void __launch_bounds__(PARSE_BLOCK) k_parse_newline_count(const __grid_constant__ ParseParams P) {
    const int64_t c = (int64_t)blockIdx.x * (PARSE_BLOCK / 32) + (threadIdx.x >> 5);
    if (c >= P.chunks) return;
    const int lane = threadIdx.x & 31;
    int n = 0;
#pragma unroll
    for (int r = 0; r < PARSE_ROUNDS; ++r) n += parse_nl16(parse_load16(P, c * PARSE_CHUNK + r * 512 + lane * 16));
    n = __reduce_add_sync(0xFFFFFFFFu, n);
    if (lane == 0) P.chunk_newlines[c] = (uint32_t)n;
}

// starts[k + 1] = one past the k-th newline; starts[0] = 0 and starts[lines] = bytes + 1 (a newline after the end)
__global__ void __launch_bounds__(PARSE_BLOCK) k_parse_line_starts(const __grid_constant__ ParseParams P) {
    const int64_t c = (int64_t)blockIdx.x * (PARSE_BLOCK / 32) + (threadIdx.x >> 5);
    if (c >= P.chunks) return;
    const int lane = threadIdx.x & 31;
    long long base = P.newlines_before[c];
    for (int r = 0; r < PARSE_ROUNDS; ++r) {
        const int64_t pos = c * PARSE_CHUNK + r * 512 + lane * 16;
        const uint4 v = parse_load16(P, pos);
        const int n = parse_nl16(v);
        int incl = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += y;
        }
        long long k = base + incl - n;
        const uint32_t m[4] = {parse_nl4(v.x), parse_nl4(v.y), parse_nl4(v.z), parse_nl4(v.w)};
#pragma unroll
        for (int b = 0; b < 16; ++b)
            if ((m[b >> 2] >> (8 * (b & 3))) & 1u) P.starts[++k] = pos + b + 1;
        base += __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    if (lane == 0 && c == 0) P.starts[0] = 0;
    if (lane == 0 && c == P.chunks - 1) P.starts[P.lines] = P.bytes + 1;
}

__global__ void __launch_bounds__(PARSE_BLOCK) k_parse_lines(const __grid_constant__ ParseParams P) {
    const int64_t i = (int64_t)blockIdx.x * PARSE_BLOCK + threadIdx.x;
    if (i < P.lines) parse_check_line(P, i);
}
__global__ void __launch_bounds__(PARSE_BLOCK) k_parse_values(const __grid_constant__ ParseParams P) {
    const int64_t i = (int64_t)blockIdx.x * PARSE_BLOCK + threadIdx.x;
    if (i < P.lines) parse_values_line(P, i);
}

}  // namespace

int launch_publish(const long long* total, const int32_t* flag, long long* mapped_dst, void* stream) {
    k_publish<<<1, 1, 0, (cudaStream_t)stream>>>(total, flag, mapped_dst);
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int launch_expand_events(const DevModel& M, const uint32_t* words, const uint8_t* dts, void* rows, long long first, long long count,
                         const EventFormat& fm, void* stream) {
    if (count <= 0) return 0;
    k_expand_events<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(M, words, dts, (uint2*)rows, first, count, fm);
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

long long scan_scratch_len(long long n) { return (n + SCAN_TILE - 1) / SCAN_TILE + 1; }

int launch_scan_counts(const uint32_t* counts, long long* offsets, long long n, long long* scratch, void* stream,
                       const long long* carry_in) {
    const long long tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    cudaStream_t st = (cudaStream_t)stream;
    k_scan_tile_sums<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(counts, scratch, n);
    k_scan_tile_prefix<<<1, 1024, 0, st>>>(scratch, tiles, offsets + n, carry_in);
    k_scan_apply<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(counts, scratch, offsets, n);
    g_launch_count.fetch_add(3);
    return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
template <class VT>
static int launch_initial_t(const DevModel& M, const SampleParams& P, int table_words, int8_t* bins, VT* values,
                            uint16_t* attempts, unsigned long long* hist, int32_t* status, void* stream) {
    if (P.n <= 0) return 0;
    const bool f32 = sizeof(VT) == 4;
    if (!g_force_generic && !hist && initial_fast_ok(M, P) && (!f32 || !values || M.init32_ok)) {
        InitStrides st;
        fill_init_strides(M, table_words, EMB_INIT_PAD, st);
        InitCalls ic;
        fill_init_calls(P, M.n_initial, ic);
        const int64_t need = (P.n + 256 * INIT_SPT - 1) / (256 * INIT_SPT);
        size_t tbytes = (size_t)st.words * 4;
        const bool smem = table_words > 0 && tbytes <= 96 * 1024 && need >= 2 * 148;   // staging pays only for large batches
        if (!smem) {
            fill_init_strides(M, table_words, 0, st);
            tbytes = (size_t)table_words * 4;
        }
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        bool done = false;
#define EMB_LAUNCH_INIT(NV_, VAL_, SM_)                                                                          \
    do {                                                                                                         \
        auto kern = (P.first_sample & 3) ? k_initial_fast<NV_, VAL_, SM_, VT, false> : k_initial_fast<NV_, VAL_, SM_, VT, true>; \
        unsigned g4 = (unsigned)need;                                                                            \
        if (SM_) {   /* persistent grid: one table copy per resident block */                                    \
            int occ = 1;                                                                                         \
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tbytes);                \
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, tbytes);                              \
            g4 = (unsigned)std::min<int64_t>(need, (int64_t)sms * std::max(occ, 1));                             \
        }                                                                                                        \
        kern<<<g4, 256, SM_ ? tbytes : 0, (cudaStream_t)stream>>>(M, P, st, ic, table_words, bins, values, attempts); \
    } while (0)
#define EMB_X(NV_)                                                          \
    if (!done && M.n_initial == (NV_)) {                                    \
        if (values && smem) EMB_LAUNCH_INIT(NV_, true, true);               \
        else if (values) EMB_LAUNCH_INIT(NV_, true, false);                 \
        else if (smem) EMB_LAUNCH_INIT(NV_, false, true);                   \
        else EMB_LAUNCH_INIT(NV_, false, false);                            \
        done = true;                                                        \
    }
        EMB_INIT_SHAPES(EMB_X)
#undef EMB_X
#undef EMB_LAUNCH_INIT
        if (done) {
            g_last_kernel_fast = 1;
            g_launch_count.fetch_add(1);
            return (int)cudaGetLastError();
        }
    }
    g_last_kernel_fast = 0;
    const unsigned grid = (unsigned)((P.n + BLOCK - 1) / BLOCK);
    k_initial<VT><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, bins, values, attempts, hist, status);
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int launch_initial(const DevModel& M, const SampleParams& P, int table_words, int8_t* bins, double* values,
                   uint16_t* attempts, unsigned long long* hist, int32_t* status, void* stream) {
    return launch_initial_t<double>(M, P, table_words, bins, values, attempts, hist, status, stream);
}
int launch_initial_f32(const DevModel& M, const SampleParams& P, int table_words, int8_t* bins, float* values,
                       uint16_t* attempts, unsigned long long* hist, int32_t* status, void* stream) {
    return launch_initial_t<float>(M, P, table_words, bins, values, attempts, hist, status, stream);
}

int launch_tracks(const DevModel& M, const SampleParams& P0, const TrackOut& O, void* stream) {
    if (P0.n <= 0) return 0;
    const uint32_t rs = g_force_generic ? 0u : fast_shape_of(M);
    const bool fast = M.fast != 0;
    const uint32_t ord = order_code(M);
    const bool hist = O.hist_initial || O.hist_transition;
    const int ev = O.ev_counts ? 1 : O.ev_words ? 2 : (O.x.xyz || O.x.is_good) ? 3 : 0;   // event / fused passes never carry histograms (emb_api.cpp)
    bool done = false;
    // one launch per run of tracks whose global sample index shares its high word (spec v5: counter word 0 is launch-uniform);
    // the last launch also covers the padding tracks up to the end of the last tile, which it zeroes (event passes skip them)
    SampleParams P = P0;
    for (int64_t s0 = 0; s0 < P0.n; s0 = P.s_end) {
        P.s_begin = s0;
        P.s_end = next_segment(P0.first_sample, s0, P0.n);
        const int64_t s_last = P.s_end == P0.n ? num_tiles(P0.n) * TRACK_TILE : P.s_end;
        const unsigned grid = (unsigned)((s_last - P.s_begin + BLOCK - 1) / BLOCK);
        done = false;
#define EMB_X(RS_, NG_, FAST_, ORD_)                                                                    \
    if (!done && rs == (RS_) && M.n_gated == (NG_) && fast == (FAST_) && ord == (ORD_)) {               \
        if (ev == 1) k_tracks_fast<RS_, NG_, FAST_, false, 1, ORD_><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O);      \
        else if (ev == 2) k_tracks_fast<RS_, NG_, FAST_, false, 2, ORD_><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O); \
        else if (ev == 3) k_tracks_fast<RS_, NG_, FAST_, false, 3, ORD_><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O); \
        else if (hist) k_tracks_fast<RS_, NG_, FAST_, true, 0, ORD_><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O);     \
        else k_tracks_fast<RS_, NG_, FAST_, false, 0, ORD_><<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O);              \
        done = true;                                                                                    \
    }
        EMB_FAST_SHAPES(EMB_X)
#undef EMB_X
        if (!done && ev == 3) return -1;   // no fused kernel for this model shape: the caller integrates in a second pass
        if (!done) k_tracks_generic<<<grid, BLOCK, 0, (cudaStream_t)stream>>>(M, P, O);
        g_launch_count.fetch_add(1);
    }
    g_last_kernel_fast = done ? 1 : 0;
    return (int)cudaGetLastError();
}


int launch_loglik_initial(const DevModel& M, const LoglikParams& P, int table_len, void* stream) {
    if (P.n <= 0) return 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t need = (P.n + 255) / 256;
    const size_t tbytes = (size_t)table_len * 8;
    const bool smem = table_len > 0 && tbytes <= 96 * 1024 && need >= 2 * sms;   // staging pays only for large batches
    unsigned grid = (unsigned)std::min<int64_t>(need, (int64_t)sms * 32);
    if (smem) {
        int occ = 1;
        cudaFuncSetAttribute(k_loglik_initial<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tbytes);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_loglik_initial<true>, 256, tbytes);
        grid = (unsigned)std::min<int64_t>(need, (int64_t)sms * std::max(occ, 1));
        k_loglik_initial<true><<<grid, 256, tbytes, (cudaStream_t)stream>>>(M, P, table_len);
    } else {
        k_loglik_initial<false><<<grid, 256, 0, (cudaStream_t)stream>>>(M, P, table_len);
    }
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

// tracks per block of the frozen-branch scoring kernels: 128 while the counters fit 96 KB of shared memory, fewer otherwise
// (8 variables of 127 bins at 32: 127 KB)
static int loglik_frozen_block(const DevModel& M) {
    const size_t per_thread = (size_t)loglik_counters(M) * 4;
    int block = 128;
    while (block > 32 && per_thread * block > 96 * 1024) block /= 2;
    return block;
}

int launch_loglik_tracks(const DevModel& M, const LoglikParams& P, void* stream) {
    if (P.n <= 0) return 0;
    if (M.fast) {
        const int block = loglik_frozen_block(M);
        const size_t bytes = (size_t)loglik_counters(M) * 4 * block;
        cudaFuncSetAttribute(k_loglik_tracks<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        k_loglik_tracks<true><<<(unsigned)((P.n + block - 1) / block), block, bytes, (cudaStream_t)stream>>>(M, P);
    } else {
        k_loglik_tracks<false><<<(unsigned)((P.n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(M, P);
    }
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

template <bool PACKED>
static void launch_loglik_events_t(const DevModel& M, const LoglikParams& P, const EventRows& R, cudaStream_t stream) {
    if (M.fast) {
        const int block = loglik_frozen_block(M);
        const size_t bytes = (size_t)loglik_counters(M) * 4 * block;
        cudaFuncSetAttribute(k_loglik_events<PACKED, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        k_loglik_events<PACKED, true><<<(unsigned)((P.n + block - 1) / block), block, bytes, stream>>>(M, P, R);
    } else {
        k_loglik_events<PACKED, false><<<(unsigned)((P.n + 127) / 128), 128, 0, stream>>>(M, P, R);
    }
}

int launch_loglik_events(const DevModel& M, const LoglikParams& P, const EventRows& R, bool packed, void* stream) {
    if (P.n <= 0) return 0;
    if (packed) launch_loglik_events_t<true>(M, P, R, (cudaStream_t)stream);
    else launch_loglik_events_t<false>(M, P, R, (cudaStream_t)stream);
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int launch_events_expand(const DevModel& M, const ExpandParams& P, const EventRows& R, bool packed, bool count, void* stream) {
    if (P.n <= 0) return 0;
    const unsigned grid = (unsigned)((P.n + EE_BLOCK / 32 - 1) / (EE_BLOCK / 32));
    cudaStream_t st = (cudaStream_t)stream;
    if (count) {
        if (packed) k_events_expand_count<true><<<grid, EE_BLOCK, 0, st>>>(M, P, R);
        else k_events_expand_count<false><<<grid, EE_BLOCK, 0, st>>>(M, P, R);
    } else {
        if (packed) k_events_expand<true><<<grid, EE_BLOCK, 0, st>>>(M, P, R);
        else k_events_expand<false><<<grid, EE_BLOCK, 0, st>>>(M, P, R);
    }
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int launch_format_csv(const CsvParams& P, bool count, void* stream) {
    if (P.n <= 0) return 0;
    const unsigned grid = (unsigned)((P.n + FMT_BLOCK / 32 - 1) / (FMT_BLOCK / 32));
    if (count) k_format_csv_count<<<grid, FMT_BLOCK, 0, (cudaStream_t)stream>>>(P);
    else k_format_csv<<<grid, FMT_BLOCK, 0, (cudaStream_t)stream>>>(P);
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int64_t parse_chunk_bytes() { return PARSE_CHUNK; }

int launch_parse(const ParseParams& P, int pass, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t items = pass < 2 ? (P.chunks + PARSE_BLOCK / 32 - 1) / (PARSE_BLOCK / 32) : (P.lines + PARSE_BLOCK - 1) / PARSE_BLOCK;
    if (items <= 0) return 0;
    const unsigned grid = (unsigned)items;
    switch (pass) {
        case 0: k_parse_newline_count<<<grid, PARSE_BLOCK, 0, st>>>(P); break;
        case 1: k_parse_line_starts<<<grid, PARSE_BLOCK, 0, st>>>(P); break;
        case 2: k_parse_lines<<<grid, PARSE_BLOCK, 0, st>>>(P); break;
        default: k_parse_values<<<grid, PARSE_BLOCK, 0, st>>>(P); break;
    }
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

int launch_format(const FormatParams& P, bool transition, bool count, void* stream) {
    if (P.n <= 0) return 0;
    const unsigned grid = (unsigned)((P.n + FMT_BLOCK / 32 - 1) / (FMT_BLOCK / 32));
    cudaStream_t st = (cudaStream_t)stream;
    if (transition) {
        if (count) k_format_transition_count<<<grid, FMT_BLOCK, 0, st>>>(P);
        else k_format_transition<<<grid, FMT_BLOCK, 0, st>>>(P);
    } else {
        if (count) k_format_initial_count<<<grid, FMT_BLOCK, 0, st>>>(P);
        else k_format_initial<<<grid, FMT_BLOCK, 0, st>>>(P);
    }
    g_launch_count.fetch_add(1);
    return (int)cudaGetLastError();
}

}  // namespace emb
