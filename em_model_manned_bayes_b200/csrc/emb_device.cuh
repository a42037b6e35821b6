// emb_device.cuh -- device-side model layout, keyed Philox stream and the per-sample sampling
// routines shared by all kernels.  Everything here is integer work except de-discretisation.
//
// Word-space inverse CDF ("normalised cumulative CPT"): for a column of weights w (N + alpha,
// select_random.m:17-20) the reference picks the first bin m with cumsum(w)(m) >= sum(w)*u.  With
// u = (k + 0.5) 2^-32 for a 32-bit Philox word k, "bin > m" is monotone in k, so the packer
// (emb_model.cpp: pack_column) stores K_m = min{k : cumsum(w)(m) < fl(sum(w) * u_k)}, found with the
// reference's own fp64 comparison.  A column occupies rp = 4*ceil(r/4) uint32 slots:
//     slots 0 .. rp-2 : T'_m = K_m - 1   (0xFFFFFFFF when K_m == 0 or K_m == 2^32 or m >= r-1)
//     slot  rp-1      : lead = #{m : K_m == 0}
// and the 0-based bin is  lead + #{m < rp-1 : k > T'_m}.   Bit-identical to the fp64 rule.
//
// The functions are __host__ __device__ only so that tests/emu can run the *same* code on the CPU
// against the oracle when no GPU is present; libemb200.so never executes them on the host.
#pragma once
#include <cmath>
#include <cstdint>

#include <vector_types.h>   // uint2 / uint4 (host and device)

#if defined(__CUDACC__)
#define EMB_HD __host__ __device__ __forceinline__
#else
#define EMB_HD inline
#endif

namespace emb {

constexpr int MAXV = 24;  // EMB_MAX_VARS
constexpr int MAXD = 8;   // EMB_MAX_DYN
constexpr int MAXP = 8;   // EMB_MAX_PARENTS
constexpr int MAXG = 16;  // EMB_MAX_GATED
constexpr int MAXX = MAXV + MAXD;
constexpr int HIST_STRIDE = 64;

// stream spec v5 (oracle/philox.py): counter = (sample >> 32, sample & 0xffffffff, attempt << 16 | purpose << 8 | sub, index);
// the step stream (P_STEP) carries no attempt: the rejection test only reads the initial draw (UncorEncounterModel.m:275),
// so the seconds of the accepted attempt are the same words whichever attempt was accepted.
constexpr uint32_t P_INIT = 1, P_STEP = 2, P_LAYER = 4;
// one word k(e, g) per (second e, gated variable g); one Philox call = four consecutive seconds of ONE variable
// (index (e >> 2) * nw + g, lane e & 3).  Select on k, gate on k*GATE_MULT; the de-discretisation word is k*DD_MULT + k',
// k' = the same variable's word of the cyclically next second of the call, which makes the value independent of the
// variable's own select and gate decisions of that second
constexpr uint32_t GATE_MULT = 0x9E3779B1u;
constexpr uint32_t DD_MULT = 0x85EBCA6Bu;

struct Node {
    int32_t r;               // bins
    int32_t rp;              // padded column length (multiple of 4)
    int32_t np;              // number of parents
    uint32_t off;            // offset of column 0 in the threshold table (uint32 units)
    uint8_t par[MAXP];       // parent indices into the state vector x (increasing)
    uint32_t stride_rp[MAXP];// asub2ind stride of that parent times rp
};

struct DevModel {
    int32_t n_initial, n_transition, n_dyn, n_gated, n_tv, nw, fast;
    int32_t order_initial[MAXV];   // 0-based ids, topological
    int32_t order_dyn[MAXD];       // dynamic ordinals in order_transition order
    Node init[MAXV];
    Node dyn[MAXD];
    int32_t dyn_t[MAXD];           // x index of the variable at time t
    int32_t dyn_t1[MAXD];          // x index of its (t+1)/(t-1) counterpart
    int32_t gated_var[MAXG];       // variables with a word per second: rate > 0 or dynamic, ascending (spec v5)
    uint64_t gate_G[MAXG];         // fires iff k*GATE_MULT mod 2^32 < G (0 for rate 0)
    int32_t gate_of_dyn[MAXD];     // gated ordinal of the d-th dynamic variable
    int32_t dd_off[MAXG];          // first entry of gated ordinal g in dd32
    int32_t ddi_off[MAXV];         // first entry of initial variable i in dd32 (entries of ALL initial variables follow the gated ones)
    int32_t init32_ok;             // every bin of every initial variable can be de-discretised in fp32 within 1e-6 relative
    int32_t fast32_ok;             // every gated bin can be de-discretised in fp32 within 1e-6 relative
    int32_t two23;                 // 2^23 as a run-time value (keeps IMAD.HI from being strength-reduced)
    int32_t tv_var[MAXV];          // time-varying variables (dynamic(t) or gated), ascending
    int32_t tv_of_var[MAXV];       // inverse map or -1
    int32_t edge_off[MAXV];        // offset (doubles) into edges of {a,w} pairs, -1 = no boundaries
    int32_t zero_bin[MAXV];        // 1-based zero bin or 0
    const uint32_t* thr_init;
    const uint32_t* thr_trans;
    const double* edges;
    const float* dd32;             // per (gated ordinal, bin): {slope, base, s, c}  (emb_model.cpp: pack)
    const double* logp_init;       // log(w_m / W) at the slots of thr_init / thr_trans; set by the scoring entry points only
    const double* logp_trans;
};

struct SampleParams {
    uint64_t seed;
    uint64_t first_sample;
    int64_t n;
    int64_t s_begin, s_end;        // tracks [s_begin, s_end) of [0, n) handled by this launch (track kernels): a launch never
                                   // straddles a multiple of 2^32 of the global sample index, so that counter word 0 of the
                                   // step stream is the same for all its tracks (spec v5; next_segment below)
    int32_t T;
    int32_t reject_mode;           // EMB_REJECT_*
    int32_t idx_v, idx_dh, idx_L;  // 0-based, -1 if unused
    int32_t is_quantize500;
    int32_t n_layers;
    int32_t max_attempts;
    uint32_t rk[20];               // Philox round keys (k0 + i*W0, k1 + i*W1), read from the constant bank
    uint8_t start[MAXV];           // preset 1-based bin, 0 = free
    const int8_t* start_ps;        // per-sample presets [n_initial][start_stride] (device memory) or nullptr
    int64_t start_stride;
    double layers[8][2];
    double box_lo[MAXV], box_hi[MAXV];
};

// Dense output layout (emb200.h: emb_track_out): tiles of TRACK_TILE tracks x four seconds, all variables of a tile together:
//     [ceil(T/4)][ceil(n/128)][var][128][4]
// so that one thread's stores of a four-second group sit at compile-time offsets (var * 128 * 4 elements) from a single running
// pointer, a warp still writes 128 (int8) or 512 (fp32) contiguous bytes per variable, and the pointer advances by one uniform
// stride per group.  (The former [var][ceil(T/4)][n][4] layout cost two 64-bit adds per store.)
constexpr int TRACK_TILE = 128;
EMB_HD int64_t num_tiles(int64_t n) { return (n + TRACK_TILE - 1) / TRACK_TILE; }
// element offset of (variable var of nvar, group grp, track s, second 0 of the group)
EMB_HD int64_t tile_offset(int nvar, int64_t ntile, int var, int64_t grp, int64_t s) {
    return (((grp * ntile + s / TRACK_TILE) * nvar + var) * TRACK_TILE + s % TRACK_TILE) * 4;
}

// zeros for padding track s (n <= s < 128 * ceil(n/128)) of the dense outputs, so that the buffers are fully defined
template <class TO>
EMB_HD void zero_padding_track(const TO& O, int nd, int ng, int T, int64_t N, int64_t s) {
    const int64_t ntile = num_tiles(N);
    if (s < N || s >= ntile * TRACK_TILE) return;
    for (int grp = 0; grp < (T + 3) >> 2; ++grp) {
        if (O.values)
            for (int g = 0; g < ng; ++g)
                for (int j = 0; j < 4; ++j) O.values[tile_offset(ng, ntile, g, grp, s) + j] = 0.0f;
        if (O.bins)
            for (int d = 0; d < nd; ++d)
                for (int j = 0; j < 4; ++j) O.bins[tile_offset(nd, ntile, d, grp, s) + j] = 0;
    }
}

// end of the segment that starts at track s0: the largest s1 <= n with (first_sample + s) >> 32 constant on [s0, s1)
inline int64_t next_segment(uint64_t first_sample, int64_t s0, int64_t n) {
    const uint64_t a = first_sample + (uint64_t)s0;
    const uint64_t room = 0x100000000ull - (a & 0xFFFFFFFFull);   // samples left before the next multiple of 2^32
    return (uint64_t)(n - s0) <= room ? n : s0 + (int64_t)room;
}

// fused first-order integration (emb_fast.cuh, mode 3 of k_tracks_fast): the Euler loop of sample2track.m:199-244 on the values of a
// group of four seconds while they are still in registers; same fields and meaning as IntegrateParams (emb_integrate.cuh)
struct XyzOut {
    float* xyz;                    // [3][T+1][n]  x_ft, y_ft, z_ft at time_s = 0..T (nullable)
    uint8_t* is_good;              // [n]  ~is_cfit & ~is_reject_speed (nullable)
    int32_t g_acc, g_vr, g_turn;   // ordinals of \dot v, \dot h, \dot\psi among the time-varying variables
    int32_t i_alt, i_speed;        // 0-based initial variables: altitude layer value, airspeed
    double ur_speed, ur_vertrate, ur_heading, min_speed, max_speed;
};

struct TrackOut {
    int8_t* bins;
    float* values;
    int8_t* init_bins;
    double* init_values;
    uint16_t* attempts;
    unsigned long long* hist_initial;
    unsigned long long* hist_transition;
    int32_t* status;               // device flag: set to 1 if any sample exhausted max_attempts
    // sparse event list (emb200.h: emb_event), two passes: count rows per track, then write them
    uint32_t* ev_counts;           // pass 1: [n] rows of each track (including the closing row)
    const long long* ev_offsets;   // pass 2: [n] first row of each track
    uint32_t* ev_words;            // pass 2: packed rows (pack_event_word below), one word and
    uint8_t* ev_dts;               //         ev_fmt.dt_bytes bytes per row
    int32_t ev_gord_bits, ev_dt_bytes;   // EventFormat of the write pass
    int64_t init_stride;           // samples between consecutive variables of init_bins / init_values; 0 = P.n (a chunk of
                                   // a larger call writes into the whole call's [n_initial][n] arrays)
    XyzOut x;                      // fused integration (both pointers null: off)
};

// ---- packed event rows: what the write pass produces and emb_sample_track_events_packed returns --------------------------------
// word = frac | (bin - 1) << 23 | gord << 27 | (dt >> 8*dt_bytes) << (27 + gord_bits);  dts = the low dt_bytes bytes of dt
//   frac : the 23 bits of the de-discretisation word, u_dd = (frac + 0.5) 2^-23 (stream spec v5) -- the value is
//          boundaries[bin] + (boundaries[bin+1] - boundaries[bin]) * u_dd, 0 in a zero bin, the bin itself for a '*' variable
//   gord : 1-based ordinal of the variable among the gated variables, 0 in the closing row (then bin and frac are 0)
//   dt   : seconds since the previous row
// The public packed format is (gord_bits, dt_bytes) = (3, 1): 5 bytes per row, n_gated <= 7, T <= 1023 -- every shipped model.
// The 8-byte emb_event rows of emb_sample_track_events are expanded from packed rows on the device (expand_event) and also
// accept 4-bit ordinals and 2-byte dts (n_gated <= 15, T <= 65535); bins of gated variables must be <= 16.
struct EventFormat {
    int32_t gord_bits, dt_bytes;
};
inline bool event_format_for(int n_gated, int max_bins, int T, EventFormat& f) {
    if (n_gated > 15 || max_bins > 16) return false;
    f.gord_bits = n_gated <= 7 ? 3 : 4;
    f.dt_bytes = T < (1 << (8 + 5 - f.gord_bits)) ? 1 : 2;
    return T < (1 << (16 + 5 - f.gord_bits));
}
EMB_HD uint32_t pack_event_word(uint32_t dt, uint32_t gord, uint32_t bin1, uint32_t frac, const EventFormat& f) {
    return frac | ((bin1 ? bin1 - 1u : 0u) << 23) | (gord << 27) | ((dt >> (8 * f.dt_bytes)) << (27 + f.gord_bits));
}
EMB_HD void store_event(uint32_t* words, uint8_t* dts, long long i, uint32_t dt, uint32_t gord, uint32_t bin1, uint32_t frac,
                        const EventFormat& f) {
    words[i] = pack_event_word(dt, gord, bin1, frac, f);
    if (f.dt_bytes == 1) dts[i] = (uint8_t)(dt & 255u);
    else reinterpret_cast<uint16_t*>(dts)[i] = (uint16_t)(dt & 65535u);
}

// ---------------------------------------------------------------------------------------------
// exact fp64 helpers (no FMA contraction, round-to-nearest) so host emulation == device
EMB_HD double dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b;
    return r;
#endif
}
EMB_HD double dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b;
    return r;
#endif
}
// u = (k + 0.5) * 2^-32, exact.  On the device k + 0.5 comes from the 2^52 trick (the word placed under the high word of 2^52,
// minus 2^52 - 0.5: one exact DADD) instead of the quarter-rate I2F.F64.U32 conversion; the value is the same double.
EMB_HD double u01(uint32_t k) {
#if defined(__CUDA_ARCH__)
    return dmul(dadd(__hiloint2double(0x43300000, (int)k), -4503599627370495.5), 2.3283064365386963e-10);
#else
    return dmul(dadd((double)k, 0.5), 2.3283064365386963e-10);
#endif
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11)
constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u, PHILOX_W1 = 0xBB67AE85u;

// 32x32 -> 64 multiply as ONE IMAD.WIDE.U32 (the C++ form is lowered through a 64-bit multiply that
// leaves a dead add per product in SASS)
EMB_HD void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    uint64_t p;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(a), "r"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(p));
#else
    const uint64_t p = (uint64_t)a * b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
#endif
}

EMB_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                          uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t h0, l0, h1, l1;
        mulhilo(PHILOX_M0, c0, h0, l0);
        mulhilo(PHILOX_M1, c2, h1, l1);
        c0 = h1 ^ c1 ^ k0;
        c2 = h0 ^ c3 ^ k1;
        c1 = l1;
        c3 = l0;
        k0 += PHILOX_W0;
        k1 += PHILOX_W1;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

// same function with the ten round keys precomputed (SampleParams::rk lives in the constant bank, so the
// key injection is a constant operand of the LOP3 and costs no instruction)
EMB_HD void philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t (&rk)[20],
                             uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t h0, l0, h1, l1;
        mulhilo(PHILOX_M0, c0, h0, l0);
        mulhilo(PHILOX_M1, c2, h1, l1);
        c0 = h1 ^ c1 ^ rk[2 * i];
        c2 = h0 ^ c3 ^ rk[2 * i + 1];
        c1 = l1;
        c3 = l0;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

// ---- the same function split by what its first three rounds depend on ------------------------------------------------
// With the spec-v4 counter (c0, c1, c2, c3) = (sample_hi, sample_lo, purpose word, index) and c0, c2 the same for every track
// of a launch, round 0 multiplies constants, round 1 multiplies one track-invariant word (M0 * a0, a0 from sample_lo) and one
// word that only depends on the index (M1 * a2), and so does round 2 -- only from round 3 on do the products depend on both.
// A track therefore keeps three words (PhiloxTrack), every call index has three words that all tracks share (philox_call:
// computed once per block into shared memory), and a call costs 7 rounds = 14 IMAD.WIDE instead of 20.  The result is
// bit-for-bit philox4x32_10(c0, c1, c2, c3) (tests/test_oracle_kat.py checks the split against the plain function).
struct PhiloxTrack {
    uint32_t r1h, r1l, q0l;
};
EMB_HD PhiloxTrack philox_track(uint32_t c0, uint32_t c1, uint32_t c2, const uint32_t (&rk)[20]) {
    uint32_t p0h, p0l, p1h, p1l, q0h, q0l;
    mulhilo(PHILOX_M0, c0, p0h, p0l);
    mulhilo(PHILOX_M1, c2, p1h, p1l);
    const uint32_t a0 = p1h ^ c1 ^ rk[0];
    mulhilo(PHILOX_M0, a0, q0h, q0l);
    const uint32_t b2 = q0h ^ p0l ^ rk[3];
    PhiloxTrack t;
    mulhilo(PHILOX_M1, b2, t.r1h, t.r1l);
    t.q0l = q0l;
    return t;
}
// x = q1l ^ rk4, y = r0h ^ rk5, z = r0l (w unused)
EMB_HD uint4 philox_call(uint32_t c0, uint32_t c2, uint32_t index, const uint32_t (&rk)[20]) {
    uint32_t p0h, p0l, p1h, p1l, q1h, q1l, r0h, r0l;
    mulhilo(PHILOX_M0, c0, p0h, p0l);
    mulhilo(PHILOX_M1, c2, p1h, p1l);
    const uint32_t a2 = p0h ^ index ^ rk[1];
    mulhilo(PHILOX_M1, a2, q1h, q1l);
    const uint32_t b0 = q1h ^ p1l ^ rk[2];
    mulhilo(PHILOX_M0, b0, r0h, r0l);
    uint4 e;
    e.x = q1l ^ rk[4];
    e.y = r0h ^ rk[5];
    e.z = r0l;
    e.w = 0;
    return e;
}
EMB_HD void philox_finish(const PhiloxTrack& t, const uint4& e, const uint32_t (&rk)[20],
                          uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
    uint32_t c0 = t.r1h ^ e.x, c1 = t.r1l, c2 = e.y ^ t.q0l, c3 = e.z;
#ifndef EMB_PHILOX_ROUNDS   // measurement only (DESIGN.md section 5): the stream spec, the oracle and every golden are 10 rounds
#define EMB_PHILOX_ROUNDS 10
#endif
#pragma unroll
    for (int i = 3; i < EMB_PHILOX_ROUNDS; ++i) {
        uint32_t h0, l0, h1, l1;
        mulhilo(PHILOX_M0, c0, h0, l0);
        mulhilo(PHILOX_M1, c2, h1, l1);
        c0 = h1 ^ c1 ^ rk[2 * i];
        c2 = h0 ^ c3 ^ rk[2 * i + 1];
        c1 = l1;
        c3 = l0;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

// Sequential reader of one (sample, attempt, purpose) word stream: position p -> block p/4, lane p%4.
// Caches the last block, so monotone access costs one Philox call per 4 words.
struct WordStream {
    uint32_t k0, k1, c0, c1, w3;
    uint32_t blk;
    uint32_t w[4];
    EMB_HD void init(uint64_t seed, uint64_t sample, uint32_t attempt, uint32_t purpose) {
        k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32);
        c0 = (uint32_t)(sample >> 32); c1 = (uint32_t)sample;
        w3 = (attempt << 16) | (purpose << 8);
        blk = 0xFFFFFFFFu;
    }
    EMB_HD uint32_t at(uint32_t p) {
        const uint32_t b = p >> 2;
        if (b != blk) {
            blk = b;
            philox4x32_10(c0, c1, w3, b, k0, k1, w[0], w[1], w[2], w[3]);
        }
        const uint32_t l = p & 3u;
        return l == 0 ? w[0] : l == 1 ? w[1] : l == 2 ? w[2] : w[3];
    }
};

EMB_HD uint32_t keyed_word(uint64_t seed, uint64_t sample, uint32_t attempt, uint32_t purpose, uint32_t index,
                           uint32_t sub, uint32_t lane) {
    uint32_t o0, o1, o2, o3;
    philox4x32_10((uint32_t)(sample >> 32), (uint32_t)sample, (attempt << 16) | (purpose << 8) | sub, index,
                  (uint32_t)seed, (uint32_t)(seed >> 32), o0, o1, o2, o3);
    return lane == 0 ? o0 : lane == 1 ? o1 : lane == 2 ? o2 : o3;
}

// ---------------------------------------------------------------------------------------------
// stream spec v5: de-discretisation uniform of a step word k with partner word kn, (((k*B + kn) mod 2^32 >> 9) + 0.5) 2^-23
EMB_HD double u_dd(uint32_t k, uint32_t kn) { return dmul(dadd((double)((k * DD_MULT + kn) >> 9), 0.5), 1.1920928955078125e-07); }
// position of the step word of second e, gated ordinal g in the (sample, P_STEP) word stream (call index * 4 + lane)
EMB_HD uint32_t step_pos(uint32_t e, uint32_t g, uint32_t nw) { return (((e >> 2) * nw + g) << 2) | (e & 3u); }
// second whose word is the partner of second e
EMB_HD uint32_t partner_second(uint32_t e) { return (e & ~3u) | ((e + 1u) & 3u); }

EMB_HD uint32_t ldg32(const uint32_t* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
EMB_HD double ldg64(const double* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// one {a, b - a} edge pair (DevModel::edges holds pairs, 16-byte aligned: cudaMalloc base + even offsets) as one 16-byte load
EMB_HD void ldg_pair(const double* e, double& a, double& w) {
#if defined(__CUDA_ARCH__)
    const double2 v = __ldg(reinterpret_cast<const double2*>(e));
    a = v.x;
    w = v.y;
#else
    a = e[0];
    w = e[1];
#endif
}

// acc - [k > t] for a threshold as stored: k > t  <=>  t - k borrows (sub.cc / subc: two instructions, no compare+select)
EMB_HD uint32_t sub_gt(uint32_t acc, uint32_t k, uint32_t t) {
#if defined(__CUDA_ARCH__)
    asm("{\n\t.reg .u32 d;\n\tsub.cc.u32 d, %2, %1;\n\tsubc.u32 %0, %0, 0;\n\t}" : "+r"(acc) : "r"(k), "r"(t));
    return acc;
#else
    return acc - (k > t ? 1u : 0u);
#endif
}

// 0-based bin of word k in a packed column (rp slots, 16-byte aligned).
EMB_HD int select_bin(const uint32_t* col, int rp, uint32_t k) {
    uint32_t neg = 0, lead = 0;   // neg = minus the number of thresholds below k
    for (int q = 0; q < rp; q += 4) {
#if defined(__CUDA_ARCH__)
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(col + q));
        const uint32_t a = v.x, b = v.y, c = v.z, d = v.w;
#else
        const uint32_t a = col[q], b = col[q + 1], c = col[q + 2], d = col[q + 3];
#endif
        neg = sub_gt(sub_gt(sub_gt(neg, k, a), k, b), k, c);
        if (q + 4 < rp) neg = sub_gt(neg, k, d); else lead = d;   // last slot holds `lead`
    }
    return (int)(lead - neg);
}

// column address of a node given the state vector
EMB_HD const uint32_t* node_column(const Node& nd, const uint32_t* table, const uint8_t* x) {
    uint32_t o = nd.off;
    for (int p = 0; p < nd.np; ++p) o += nd.stride_rp[p] * (uint32_t)x[nd.par[p]];
    return table + o;
}

// dediscretize.m:22-41 for 0-based bin `b` of variable i given uniform u (only read when needed)
EMB_HD bool needs_uniform(const DevModel& M, int i, int b) {
    return M.edge_off[i] >= 0 && M.zero_bin[i] != b + 1;
}
EMB_HD double dedisc(const DevModel& M, int i, int b, double u) {
    if (M.edge_off[i] < 0) return (double)(b + 1);          // dediscretize.m:7-10: return the bin
    if (M.zero_bin[i] == b + 1) return 0.0;                 // :24-25
    double a, w;
    ldg_pair(M.edges + M.edge_off[i] + 2 * b, a, w);
    return dadd(a, dmul(w, u));                             // :39  a + (b-a)*rand
}

// packed row -> emb_event fields {dt | var << 16 | bin << 24, value as fp32 bits}.  The value is computed exactly as the
// kernel that wrote the dense output computes it: from the fp32 entry table when the model has one (emb_fast.cuh), else in
// fp64 (dediscretize.m:22-41) and rounded to fp32.
EMB_HD uint2 expand_event(const DevModel& M, uint32_t word, uint32_t dt_lo, const EventFormat& fm) {
    const uint32_t gord = (word >> 27) & ((1u << fm.gord_bits) - 1u), dt = dt_lo | ((word >> (27 + fm.gord_bits)) << (8 * fm.dt_bytes));
    uint2 row;
    if (gord == 0) {
        row.x = dt;
        row.y = 0u;
        return row;
    }
    const int g = (int)gord - 1, v = M.gated_var[g], b = (int)((word >> 23) & 15u);
    const uint32_t frac = word & 0x7FFFFFu;
    float value;
    if (M.fast32_ok) {
        const float* en = M.dd32 + 4 * (M.dd_off[g] + b);   // {slope, base, s, c}
        const uint32_t fb = frac | 0x3F800000u;
        float f;
#if defined(__CUDA_ARCH__)
        f = __uint_as_float(fb);
        value = __fmaf_rn(en[0], __fmaf_rn(f, en[2], en[3]), en[1]);
#else
        __builtin_memcpy(&f, &fb, 4);
        value = __builtin_fmaf(en[0], __builtin_fmaf(f, en[2], en[3]), en[1]);
#endif
    } else {
        value = (float)dedisc(M, v, b, dmul(dadd((double)frac, 0.5), 1.1920928955078125e-07));
    }
    row.x = dt | ((uint32_t)(v + 1) << 16) | ((uint32_t)(b + 1) << 24);
#if defined(__CUDA_ARCH__)
    row.y = __float_as_uint(value);
#else
    __builtin_memcpy(&row.y, &value, 4);
#endif
    return row;
}

EMB_HD double round500(double num) {                        // UncorEncounterModel.m:196
    double m = ::fmod(num, 500.0);
    if (m < 0) m += 500.0;
    const double q = ::floor(num / 500.0);
    return 500.0 * (q + (m > 250.0 ? 1.0 : 0.0));
}

// ---------------------------------------------------------------------------------------------
// Initial network: bn_sample.m:39-58 + dbn_hierarchical_sample.m:25-31 (+ rejection of the driver:
// UncorEncounterModel.m:248-280 / @CorTerminalModel/sample.m:32-72).
// x: 0-based bins (size >= n_transition, dynamic slots untouched); vals: continuous values.
// Returns the attempt index that was accepted, -1 when max_attempts was exhausted, -2 when this sample's presets are invalid
// (per-sample `start` rows only; the uniform `start` is validated on the host).
EMB_HD int sample_initial(const DevModel& M, const SampleParams& P, uint64_t sample, uint8_t* x, double* vals) {
    const int n = M.n_initial;
    uint8_t st[MAXV];                                                               // this sample's presets (bn_sample.m:45)
    const int64_t sl = (int64_t)(sample - P.first_sample);
    for (int i = 0; i < n; ++i) {
        int v = P.start_ps ? (int)P.start_ps[(int64_t)i * P.start_stride + sl] : (int)P.start[i];
        if (v < 0 || v > M.init[i].r) return -2;                                    // preset bin out of range
        st[i] = (uint8_t)v;
    }
    if (P.start_ps)                                                                 // bn_sample.m:46-47, per sample
        for (int i = 0; i < n; ++i)
            if (st[i])
                for (int q = 0; q < M.init[i].np; ++q)
                    if (!st[M.init[i].par[q]]) return -2;
    for (int attempt = 0; attempt <= P.max_attempts; ++attempt) {
        // stream spec v5, INIT: one word per variable; four consecutive samples share a call (sample >> 2, lane sample & 3)
        uint32_t kw[MAXV + 1];
        const int nwords = n > 1 ? n : 2;
        for (int i = 0; i < nwords; ++i)
            kw[i] = keyed_word(P.seed, sample >> 2, (uint32_t)attempt, P_INIT, (uint32_t)i, 0, (uint32_t)(sample & 3u));
        for (int oi = 0; oi < n; ++oi) {
            const int i = M.order_initial[oi];
            if (st[i]) {
                x[i] = (uint8_t)(st[i] - 1);                                        // bn_sample.m:49
            } else {
                const Node& nd = M.init[i];
                x[i] = (uint8_t)select_bin(node_column(nd, M.thr_init, x), nd.rp, kw[i]);
            }
        }
        for (int i = 0; i < n; ++i) {
            const int b = x[i];
            double u = 0.5;
            if (needs_uniform(M, i, b)) u = u_dd(kw[i], kw[i + 1 < nwords ? i + 1 : 0]);
            vals[i] = dedisc(M, i, b, u);
        }
        bool good = true;
        if (P.reject_mode == 1) {
            if (P.n_layers > 0 || P.is_quantize500) {
                double h = vals[P.idx_L];
                if (P.n_layers > 0) {                                               // UncorEncounterModel.m:259-260
                    const int L = x[P.idx_L];
                    const uint32_t k = keyed_word(P.seed, sample, (uint32_t)attempt, P_LAYER, 0, 0, 0);
                    h = dadd(P.layers[L][0], dmul(u01(k), dadd(P.layers[L][1], -P.layers[L][0])));
                }
                if (P.is_quantize500 && vals[P.idx_dh] == 0.0) h = round500(h);     // :266-268
                vals[P.idx_L] = h;                                                  // :270-272
            }
            const double a = vals[P.idx_dh] < 0 ? -vals[P.idx_dh] : vals[P.idx_dh];
            good = dmul(vals[P.idx_v], 1.68781) > a / 60.0;                         // :275
        } else if (P.reject_mode == 2) {
            for (int i = 0; i < n; ++i) good = good && (vals[i] >= P.box_lo[i]) && (vals[i] <= P.box_hi[i]);
        }
        if (good) return attempt;
    }
    return -1;
}

// ---------------------------------------------------------------------------------------------
// Generic track sampler (any model within the EMB_MAX_* limits, both dbn_sample.m branches).
// One call = one track.  Dense tiled output, see emb200.h.  `hist` (nullable) is a block-shared
// [n_dyn][HIST_STRIDE] uint32 scratch on the device.
template <class HistInc>
EMB_HD void track_generic(const DevModel& M, const SampleParams& P, const TrackOut& O, int64_t s, HistInc hist_inc) {
    uint8_t x[MAXX];
    double vals[MAXV];
    const uint64_t sample = P.first_sample + (uint64_t)s;
    const int n = M.n_initial, nd = M.n_dyn, ng = M.n_gated, nw = M.nw;
    const int T = P.T;
    const int64_t N = P.n;
    for (int i = 0; i < MAXX; ++i) x[i] = 0;

    int attempt = sample_initial(M, P, sample, x, vals);
    if (attempt < 0) {
        if (O.status) *O.status = attempt == -2 ? 2 : 1;
        attempt = P.max_attempts;  // keep the last attempt's state so the outputs are defined
    }
    if (O.attempts) O.attempts[s] = (uint16_t)(attempt + 1);
    for (int i = 0; i < n; ++i) {
        if (O.init_bins) O.init_bins[(int64_t)i * (O.init_stride ? O.init_stride : N) + s] = (int8_t)(x[i] + 1);
        if (O.init_values) O.init_values[(int64_t)i * (O.init_stride ? O.init_stride : N) + s] = vals[i];
        if (O.hist_initial) hist_inc(0, i, x[i]);
    }
    if (T <= 0 || (!O.bins && !O.values && !O.hist_transition && !O.ev_counts && !O.ev_words)) return;

    // frozen columns of the fast branch (dbn_sample.m:110-135): parents evaluated once at t = 1
    const uint32_t* col[MAXD];
    for (int d = 0; d < nd; ++d) {
        x[M.dyn_t1[d]] = x[M.dyn_t[d]];
        col[d] = node_column(M.dyn[d], M.thr_trans, x);
    }

    // event list (emb200.h: emb_event): pass 1 counts rows, pass 2 writes them
    const bool ev = O.ev_counts || O.ev_words;
    long long ev_i = O.ev_words ? O.ev_offsets[s] : 0;
    uint32_t ev_last = 0, ev_n = 0;
    // gord: 1-based gated ordinal (0 = closing row); frac: the 23 value bits of the row (see pack_event_word)
    auto emit = [&](uint32_t e, uint32_t gord, uint32_t bin1, uint32_t frac) {
        if (O.ev_words) {
            store_event(O.ev_words, O.ev_dts, ev_i, e - ev_last, gord, bin1, frac, EventFormat{O.ev_gord_bits, O.ev_dt_bytes});
            ++ev_i;
        }
        ev_last = e;
        ++ev_n;
    };

    WordStream ws;
    ws.init(P.seed, sample, 0u, P_STEP);
    const int nch4 = (T + 3) >> 2;
    uint32_t bpack[MAXD];
    float vbuf[MAXV][4];
    for (int d = 0; d < MAXD; ++d) bpack[d] = 0;

    const int Tpad = nch4 * 4;
    for (int c = 0; c < Tpad; ++c) {          // column c = state during second c+1; step e = c
        if (c > 0 && c < T) {
            uint32_t wstep[MAXG], wpart[MAXG];                  // stream spec v5: k(e, g) and its value partner k(e', g)
            for (int q = 0; q < nw; ++q) {
                wstep[q] = ws.at(step_pos((uint32_t)c, (uint32_t)q, (uint32_t)nw));
                wpart[q] = ws.at(step_pos(partner_second((uint32_t)c), (uint32_t)q, (uint32_t)nw));
            }
            // resample gates on the pre-transition bins (resample_events.m:23-29)
            for (int g = 0; g < ng; ++g) {
                const uint32_t k = wstep[g];
                if ((uint64_t)(k * GATE_MULT) < M.gate_G[g]) {
                    const int v = M.gated_var[g];
                    vals[v] = dedisc(M, v, x[v], u_dd(k, wpart[g]));
                    if (ev) emit((uint32_t)c, (uint32_t)g + 1u, (uint32_t)x[v] + 1u, (k * DD_MULT + wpart[g]) >> 9);
                }
            }
            // transitions (dbn_sample.m:69-79 slow / :143-146 fast): the variable's own word selects
            for (int od = 0; od < nd; ++od) {
                const int d = M.fast ? od : M.order_dyn[od];
                const Node& nd_ = M.dyn[d];
                const uint32_t* cp = M.fast ? col[d] : node_column(nd_, M.thr_trans, x);
                x[M.dyn_t1[d]] = (uint8_t)select_bin(cp, nd_.rp, wstep[M.gate_of_dyn[d]]);
            }
            // map back + change events (dbn_sample.m:82-92); the new value reads the same value word
            for (int d = 0; d < nd; ++d) {
                const int vt = M.dyn_t[d];
                const uint8_t nb = x[M.dyn_t1[d]];
                if (nb != x[vt]) {
                    x[vt] = nb;
                    vals[vt] = dedisc(M, vt, nb, u_dd(wstep[M.gate_of_dyn[d]], wpart[M.gate_of_dyn[d]]));
                    if (ev) emit((uint32_t)c, (uint32_t)M.gate_of_dyn[d] + 1u, (uint32_t)nb + 1u,
                                 (wstep[M.gate_of_dyn[d]] * DD_MULT + wpart[M.gate_of_dyn[d]]) >> 9);
                }
            }
        }
        const bool live = c < T;
        for (int d = 0; d < nd; ++d) {
            const uint32_t b = live ? (uint32_t)(x[M.dyn_t[d]] + 1) : 0u;
            bpack[d] |= b << (8 * (c & 3));
            if (live && c > 0 && O.hist_transition) hist_inc(1, d, x[M.dyn_t[d]]);
        }
        for (int g = 0; g < ng; ++g) vbuf[g][c & 3] = live ? (float)vals[M.gated_var[g]] : 0.0f;
        if ((c & 3) == 3) {
            if (O.values) {
                for (int g = 0; g < ng; ++g) {
                    float* dst = O.values + tile_offset(ng, num_tiles(N), g, c >> 2, s);
#if defined(__CUDA_ARCH__)
                    *reinterpret_cast<float4*>(dst) = make_float4(vbuf[g][0], vbuf[g][1], vbuf[g][2], vbuf[g][3]);
#else
                    dst[0] = vbuf[g][0]; dst[1] = vbuf[g][1]; dst[2] = vbuf[g][2]; dst[3] = vbuf[g][3];
#endif
                }
            }
            if (O.bins) {
                for (int d = 0; d < nd; ++d) {
                    int8_t* dst = O.bins + tile_offset(nd, num_tiles(N), d, c >> 2, s);
#if defined(__CUDA_ARCH__)
                    *reinterpret_cast<uint32_t*>(dst) = bpack[d];
#else
                    for (int b = 0; b < 4; ++b) dst[b] = (int8_t)((bpack[d] >> (8 * b)) & 0xFF);
#endif
                }
            }
            for (int d = 0; d < nd; ++d) bpack[d] = 0;
        }
    }
    if (ev) {
        // gates of the last held second T (resample_events.m:23-29), then the closing row (dbn_hierarchical_sample.m:15-19)
        for (int g = 0; g < ng; ++g) {
            const uint32_t k = ws.at(step_pos((uint32_t)T, (uint32_t)g, (uint32_t)nw));
            if ((uint64_t)(k * GATE_MULT) < M.gate_G[g]) {
                const int v = M.gated_var[g];
                const uint32_t kn = ws.at(step_pos(partner_second((uint32_t)T), (uint32_t)g, (uint32_t)nw));
                emit((uint32_t)T, (uint32_t)g + 1u, (uint32_t)x[v] + 1u, (k * DD_MULT + kn) >> 9);
            }
        }
        emit((uint32_t)T, 0u, 0u, 0u);
        if (O.ev_counts) O.ev_counts[s] = ev_n;
    }
}

}  // namespace emb
