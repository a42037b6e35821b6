// emb_format.cuh -- the legacy text files of em_sample.m (initial.txt, transition.txt) formatted on the device: C's "%g" of a
// double and "%d" of an int64, and the per-track routines of k_format_{initial,transition}[_count] (emb_kernels.cu); and the CSV
// rows of sample2track.m ("%.0f", k_format_csv[_count], at the end of this file).
// __host__ __device__ like emb_events_expand.cuh, so that tests/emu runs the same code on the CPU.
//
// "%g" (C99 7.19.6.1, precision 6) is defined on the exact binary value v = m * 2^e: D = the 6-digit integer nearest to
// v / 10^k, ties to even, with k = X0 - 5 and X0 = floor(log10 |v|); a carry to 10^6 gives D = 10^5 and k + 1.  X = k + 5 is the
// exponent of the rounded value, "%f" style for -4 <= X < 6 and "%e" style otherwise, trailing zeros and a bare point dropped.
// The quotient and the comparison of the remainder with half the divisor are computed in exact integer arithmetic on
// A / B = v / 10^k (A = m 2^max(e,0) 10^max(-k,0), B = 2^max(-e,0) 10^max(k,0)): in 128 bits when A and B fit in 125 bits
// (every |v| from about 1e-17 to 1e37, so every sampled value and every id), otherwise in multi-word integers of up to 1280
// bits (emb_exact.cuh; A <= 2^53 * 10^329 < 2^1147 for the subnormals, B <= 2^1074).  A double quotient only proposes q; the
// integer remainder corrects it.  Nothing is approximated, so the result is exact for every finite double (DESIGN.md section 13).
//
// Shape: one warp per track.  Lanes take consecutive items (transition: the rows of consecutive seconds; initial: the id and the
// values of the row); a warp scan of their byte lengths gives every lane its offset, the lanes move their items into the warp's
// shared-memory stage at those offsets, and the warp stores the stage as one contiguous block.  The count pass and the write pass
// emit through the same templates (fmt_emit_*, fmt_item, fmt_stage_track) into a counting or a writing sink, so their byte
// counts agree by construction.
#pragma once
#include <cstdint>

#include "emb_events_expand.cuh"   // ExpandLanes (a warp on the device, one lane in the emulation), ll_flag
#include "emb_exact.cuh"           // fmt_bits, u128, FmtBig and its operations

namespace emb {

constexpr int32_t FMT_BAD_VALUE = 1;   // status bit: a non-finite value
constexpr int FMT_G_MAX = 13;          // longest "%g" of a double: -1.23457e-308
constexpr int FMT_D_MAX = 20;          // longest "%d" of an int64
// longest transition row: id and t (%g), one " %g" per dynamic variable, "\n"; the longest initial item is shorter
constexpr int FMT_ROW_MAX = 2 * FMT_G_MAX + 1 + MAXD * (1 + FMT_G_MAX) + 1;
constexpr int FMT_STAGE = 32 * FMT_ROW_MAX;   // the packed rows of one warp's 32 lanes
constexpr int FMT_STAGE_BYTES = 2 * FMT_STAGE; // shared memory of one warp in the write pass: packed rows, then a slot per lane

struct FormatParams {
    int64_t n;
    int32_t T;
    int32_t n_initial;
    int32_t n_dyn;
    int32_t n_tv;                     // time-varying variables of the tiles
    int64_t first_id;                 // id of track 0
    const double* init_values;        // [n_initial][n] (initial text)
    const float* values;              // dense tiles [ceil(T/4)][ceil(n/128)][n_tv][128][4] (transition text)
    int32_t cols[MAXD];               // tile ordinal of each dynamic variable, temporal_map(:,1) order
    const long long* offsets;         // [n+1] bytes before each track (write pass)
    char* text;                       // write pass
    uint32_t* counts;                 // [n] bytes of each track (count pass)
    int32_t* status;                  // FMT_BAD_VALUE
};

// ---- "%g" -----------------------------------------------------------------------------------------------------------------

// v = (-1)^neg * d * 10^(x - 5), d in [10^5, 10^6), or d = 0 for a zero
struct G6 {
    uint32_t d;
    int32_t x;
    bool neg;
    bool bad;   // inf or NaN
};

EMB_HD int fmt_bitlen(u128 x) {
    const uint64_t hi = (uint64_t)(x >> 64), lo = (uint64_t)x;
    return hi ? 128 - fmt_clz64(hi) : lo ? 64 - fmt_clz64(lo) : 0;
}
EMB_HD u128 fmt_pow10(int j) {   // 10^j, j <= 38
    u128 p = 1;
    for (int i = 0; i < j; ++i) p *= 10u;
    return p;
}
EMB_HD double fmt_u128_double(u128 x) { return (double)(uint64_t)(x >> 64) * 18446744073709551616.0 + (double)(uint64_t)x; }

// q = floor(A / B) < 2^25 and the sign of 2 (A - q B) - B, from a quotient proposed in double and corrected in integers.
// The proposal is within one of q (relative error below 2^-49 on a quotient below 2^25), so one step each way suffices.
EMB_HD void fmt_divmod128(u128 A, u128 B, uint32_t& q, int& half) {
    uint32_t p = (uint32_t)(fmt_u128_double(A) / fmt_u128_double(B));
    u128 pb = B * p;   // p <= q + 1, so p B <= A + B < 2^126
    if (pb > A) {
        --p;
        pb -= B;
    }
    u128 r = A - pb;
    if (r >= B) {
        ++p;
        r -= B;
    }
    q = p;
    r <<= 1;
    half = r < B ? -1 : r > B ? 1 : 0;
}

EMB_HD void fmt_divmod_big(const FmtBig& A, const FmtBig& B, uint32_t& q, int& half) {
    double ratio = big_top(A) / big_top(B);
    for (int i = B.n; i < A.n; ++i) ratio *= 4294967296.0;
    for (int i = A.n; i < B.n; ++i) ratio *= 1.0 / 4294967296.0;
    uint32_t p = (uint32_t)ratio;
    FmtBig R = A, pb = B;
    big_mul(pb, p);
    if (big_cmp(pb, A) > 0) {
        --p;
        big_sub(pb, B);
    }
    big_sub(R, pb);
    if (big_cmp(R, B) >= 0) {
        ++p;
        big_sub(R, B);
    }
    q = p;
    big_add(R, R);
    half = big_cmp(R, B);
}

// the same outside the 128-bit range
EMB_HD void fmt_divmod_wide(uint64_t m, int ea, int eb, int ka, int kb, uint32_t& q, int& half) {
    FmtBig A, B;
    big_set(A, m);
    big_shl(A, ea);
    big_mul_pow10(A, ka);
    big_set(B, 1);
    big_shl(B, eb);
    big_mul_pow10(B, kb);
    fmt_divmod_big(A, B, q, half);
}

// floor(m 2^e / 10^k) and the sign of (remainder - divisor / 2), exactly; m odd or 1, m < 2^53
EMB_HD void fmt_divmod(uint64_t m, int e, int k, uint32_t& q, int& half) {
    const int ea = e > 0 ? e : 0, eb = e < 0 ? -e : 0, ka = k < 0 ? -k : 0, kb = k > 0 ? k : 0;
    if (ka <= 37 && kb <= 37) {
        const u128 pa = fmt_pow10(ka), pb = fmt_pow10(kb);
        const int la = 64 - fmt_clz64(m) + ea + fmt_bitlen(pa) - 1, lb = eb + fmt_bitlen(pb) - 1;   // bit lengths of A, B minus one
        if (la < 125 && lb < 125) {
            fmt_divmod128(((u128)m << ea) * pa, (u128)pb << eb, q, half);
            return;
        }
    }
    fmt_divmod_wide(m, ea, eb, ka, kb, q, half);
}


// the six significant digits and the exponent "%g" prints
EMB_HD G6 fmt_g6(double v) {
    const uint64_t bits = fmt_bits(v);
    G6 g{0u, 0, (bits >> 63) != 0, false};
    const int be = (int)((bits >> 52) & 0x7FF);
    uint64_t m = bits & 0xFFFFFFFFFFFFFull;
    if (be == 0x7FF) {
        g.bad = true;
        return g;
    }
    if (be) m |= 1ull << 52;
    if (!m) return g;
    int e = (be ? be : 1) - 1075;
    const int tz = fmt_ctz64(m);
    m >>= tz;
    e += tz;
    const int l2 = 63 - fmt_clz64(m) + e;   // floor(log2 |v|)
    // floor(l2 log10 2) is floor(log10 |v|) or one less; the loop moves k until 10^5 <= q < 10^6
    int k = (int)floor((double)l2 * 0.30102999566398120) - 5;
    uint32_t q;
    int half;
    for (;;) {
        fmt_divmod(m, e, k, q, half);
        if (q >= 1000000u) ++k;
        else if (q < 100000u) --k;
        else break;
    }
    q += (half > 0 || (half == 0 && (q & 1u))) ? 1u : 0u;
    if (q == 1000000u) {
        q = 100000u;
        ++k;
    }
    g.d = q;
    g.x = k + 5;
    return g;
}

struct FmtCount {
    int32_t n = 0;
    EMB_HD void put(char) { ++n; }
};
struct FmtWrite {
    char* p;
    EMB_HD void put(char c) { *p++ = c; }
};

template <class S>
EMB_HD void fmt_emit_g(const G6& g, S& out) {
    if (g.neg) out.put('-');
    if (!g.d) {
        out.put('0');
        return;
    }
    char dig[6];
    uint32_t d = g.d;
    for (int i = 5; i >= 0; --i) {
        dig[i] = (char)('0' + d % 10u);
        d /= 10u;
    }
    int nd = 6;
    while (dig[nd - 1] == '0') --nd;
    const int x = g.x;
    if (x >= -4 && x < 6) {
        if (x >= 0) {
            for (int i = 0; i <= x; ++i) out.put(dig[i]);
            if (nd > x + 1) {
                out.put('.');
                for (int i = x + 1; i < nd; ++i) out.put(dig[i]);
            }
        } else {
            out.put('0');
            out.put('.');
            for (int i = 0; i < -x - 1; ++i) out.put('0');
            for (int i = 0; i < nd; ++i) out.put(dig[i]);
        }
        return;
    }
    out.put(dig[0]);
    if (nd > 1) {
        out.put('.');
        for (int i = 1; i < nd; ++i) out.put(dig[i]);
    }
    out.put('e');
    out.put(x < 0 ? '-' : '+');
    const int ax = x < 0 ? -x : x;
    if (ax >= 100) out.put((char)('0' + ax / 100));
    out.put((char)('0' + ax / 10 % 10));
    out.put((char)('0' + ax % 10));
}

template <class S>
EMB_HD void fmt_emit_d(int64_t v, S& out) {
    uint64_t u = (uint64_t)v;
    if (v < 0) {
        out.put('-');
        u = 0ull - u;
    }
    char dig[FMT_D_MAX];
    int nd = 0;
    do {
        dig[nd++] = (char)('0' + u % 10u);
        u /= 10u;
    } while (u);
    while (nd) out.put(dig[--nd]);
}

// bytes of "%g" % v: the same digits and the same emitter as the text
EMB_HD int32_t fmt_g_len(double v) {
    FmtCount c;
    fmt_emit_g(fmt_g6(v), c);
    return c.n;
}

// ---- rows -------------------------------------------------------------------------------------------------------------------

// item j of track s in initial.txt: j = 0 the id ("%d"), j >= 1 " %g" of variable j-1, "\n" after the last; false if non-finite
template <class S>
EMB_HD bool fmt_initial_item(const FormatParams& P, int64_t s, int j, S& out) {
    bool ok = true;
    if (j == 0) {
        fmt_emit_d(P.first_id + s, out);
    } else {
        const G6 g = fmt_g6(P.init_values[(int64_t)(j - 1) * P.n + s]);
        ok = !g.bad;
        out.put(' ');
        fmt_emit_g(g, out);
    }
    if (j == P.n_initial) out.put('\n');
    return ok;
}

// row t of track s in transition.txt: "%g %g" of (id, t), " %g" of each dynamic variable's value in second t, "\n"
template <class S>
EMB_HD bool fmt_transition_row(const FormatParams& P, int64_t s, int t, const G6& id, S& out) {
    fmt_emit_g(id, out);
    const int64_t ntile = (P.n + 127) / 128;
    const float* tile = P.values + ((((int64_t)(t >> 2) * ntile + s / 128) * P.n_tv) * 128 + s % 128) * 4 + (t & 3);
    bool ok = true;
    for (int f = -1; f < P.n_dyn; ++f) {   // one digit generation site for t and the values keeps the kernels small
        const G6 g = fmt_g6(f < 0 ? (double)t : (double)tile[(int64_t)P.cols[f] * 512]);
        ok &= !g.bad;
        out.put(' ');
        fmt_emit_g(g, out);
    }
    out.put('\n');
    return ok;
}

template <bool TRANS, class S>
EMB_HD bool fmt_item(const FormatParams& P, int64_t s, int j, const G6& id, S& out) {
    return TRANS ? fmt_transition_row(P, s, j, id, out) : fmt_initial_item(P, s, j, out);
}

// The staging shared by every text of this file: `items` items of one track, lane j of the warp taking items j, j + W, ...;
// `item(j, sink)` emits item j (at most FMT_ROW_MAX bytes) and returns false for a non-finite value.  The count pass
// (WRITE = false) returns the track's bytes; the write pass also stores them from dst on.  stage: FMT_STAGE_BYTES of the warp's
// shared memory (write pass): a slot of FMT_ROW_MAX bytes per lane, into which the lane emits its item once, then the items
// packed at their scanned offsets, stored to global memory as one contiguous block.
template <bool WRITE, class Item>
EMB_HD uint32_t fmt_stage_track(const Item& item, int items, char* dst, const ExpandLanes& L, char* stage, bool& ok) {
    const int W = ExpandLanes::width();
    char* slot = stage + FMT_STAGE + L.lane * FMT_ROW_MAX;
    uint32_t total = 0;
    for (int base = 0; base < items; base += W) {
        const int j = base + L.lane;
        int32_t len = 0;
        if (WRITE) {
            FmtWrite w{slot};
            if (j < items) item(j, w);
            len = (int32_t)(w.p - slot);
        } else {
            FmtCount c;
            if (j < items) ok &= item(j, c);
            len = c.n;
        }
        const int32_t incl = L.scan(len);
        const int32_t chunk = L.last(incl);
        if (WRITE) {
            for (int b = 0; b < len; ++b) stage[incl - len + b] = slot[b];
            L.sync();
            for (int b = L.lane; b < chunk; b += W) dst[total + b] = stage[b];
            L.sync();
        }
        total += (uint32_t)chunk;
    }
    return total;
}

template <bool TRANS>
struct FmtEmSampleItem {
    const FormatParams& P;
    int64_t s;
    G6 id;
    template <class S>
    EMB_HD bool operator()(int j, S& out) const { return fmt_item<TRANS>(P, s, j, id, out); }
};

// Both passes of track s of initial.txt or transition.txt (fmt_stage_track).
template <bool TRANS, bool WRITE>
EMB_HD uint32_t format_track(const FormatParams& P, int64_t s, const ExpandLanes& L, char* stage) {
    const int items = TRANS ? P.T : P.n_initial + 1;
    const FmtEmSampleItem<TRANS> item{P, s, TRANS ? fmt_g6((double)(P.first_id + s)) : G6{}};
    bool ok = true;
    const uint32_t total = fmt_stage_track<WRITE>(item, items, WRITE ? P.text + P.offsets[s] : nullptr, L, stage, ok);
    if (!ok) ll_flag(P.status, FMT_BAD_VALUE);
    return total;
}

// ---- the CSV rows of sample2track.m (emb_format_tracks_csv) -------------------------------------------------------------------
// One file body per track: T+1 rows "%d,%.0f,%.0f,%.0f\n" of (t, x_ft, y_ft, z_ft), t = 0 .. T, exactly as the Python statement
// "%d,%.0f,%.0f,%.0f\n" % (t, x, y, z) formats the fp32 points widened to double.
//
// "%.0f" of a double is the integer nearest its exact value, ties to even, with "-" whenever the sign bit is set (so -0.4 and
// -0.0 print "-0").  A finite float32 f = M 2^E (M < 2^24) is decided in integers: for |f| < 2^23 (E < 0) the quotient M >> -E
// and its remainder against half of 2^-E; for |f| >= 2^23 f is an integer, M << E < 2^128, printed exactly from four 32-bit limbs
// by repeated division by 10^9 (up to 39 digits).

struct CsvParams {
    int64_t n;
    int32_t T;
    const float* xyz;                 // [3][T+1][n] (emb_tracks_integrate)
    const uint8_t* mask;              // [n] or nullptr; 0: no text for the track
    const long long* offsets;         // [n+1] bytes before each track (write pass)
    char* text;                       // write pass
    uint32_t* counts;                 // [n] bytes of each track (count pass)
    int32_t* status;                  // FMT_BAD_VALUE
};

// longest CSV row: "%d" of t < 2^31 (10 bytes), three ",-" and 39 digits (FLT_MAX), "\n"; it fits the staging slot
constexpr int FMT_CSV_ROW_MAX = 10 + 3 * (2 + 39) + 1;
static_assert(FMT_CSV_ROW_MAX <= FMT_ROW_MAX, "a CSV row must fit the staging slot of a lane");

EMB_HD uint32_t fmt_float_bits(float f) {
#if defined(__CUDA_ARCH__)
    return (uint32_t)__float_as_uint(f);
#else
    uint32_t b;
    std::memcpy(&b, &f, 4);
    return b;
#endif
}

template <class S>
EMB_HD void fmt_emit_u32(uint32_t u, S& out) {
    char dig[10];
    int nd = 0;
    do {
        dig[nd++] = (char)('0' + u % 10u);
        u /= 10u;
    } while (u);
    while (nd) out.put(dig[--nd]);
}

// "%.0f" of f widened to double; false (and nothing emitted) for inf and NaN
template <class S>
EMB_HD bool fmt_emit_f0(float f, S& out) {
    const uint32_t b = fmt_float_bits(f);
    const int be = (int)((b >> 23) & 0xFFu);
    if (be == 0xFF) return false;
    if (b >> 31) out.put('-');
    const uint32_t M = (b & 0x7FFFFFu) | (be ? 0x800000u : 0u);
    if (be < 150) {   // |f| < 2^23: f = M 2^-sh, sh = 1 .. 149
        const int sh = 150 - (be ? be : 1);
        uint32_t u = 0;
        if (sh <= 25) {   // otherwise |f| < 2^24 2^-26, which rounds to 0
            u = M >> sh;
            const uint32_t rem = M & ((1u << sh) - 1u), half = 1u << (sh - 1);
            u += (rem > half || (rem == half && (u & 1u))) ? 1u : 0u;
        }
        fmt_emit_u32(u, out);
        return true;
    }
    const u128 v = (u128)M << (be - 150);   // an integer below 2^128
    uint32_t w[4] = {(uint32_t)v, (uint32_t)(v >> 32), (uint32_t)(v >> 64), (uint32_t)(v >> 96)};
    char dig[40];
    int nd = 0;
    bool more;
    do {   // the lowest nine digits per round: w /= 10^9, r = the remainder
        uint64_t r = 0;
        for (int i = 3; i >= 0; --i) {
            const uint64_t cur = (r << 32) | w[i];
            w[i] = (uint32_t)(cur / 1000000000u);
            r = cur % 1000000000u;
        }
        more = (w[0] | w[1] | w[2] | w[3]) != 0;
        for (int k = 0; k < 9 && (more || r); ++k) {   // all nine below a higher group, no leading zeros in the top one
            dig[nd++] = (char)('0' + r % 10u);
            r /= 10u;
        }
    } while (more);
    while (nd) out.put(dig[--nd]);
    return true;
}

// row t of a track: "%d,%.0f,%.0f,%.0f\n" of (t, x, y, z); false if a coordinate is not finite
template <class S>
EMB_HD bool fmt_csv_row(const CsvParams& P, int64_t s, int t, S& out) {
    fmt_emit_d(t, out);
    const int64_t plane = (int64_t)(P.T + 1) * P.n;
    const float* p = P.xyz + (int64_t)t * P.n + s;
    bool ok = true;
    for (int c = 0; c < 3; ++c) {
        out.put(',');
        ok &= fmt_emit_f0(p[c * plane], out);
    }
    out.put('\n');
    return ok;
}

struct FmtCsvItem {
    const CsvParams& P;
    int64_t s;
    template <class S>
    EMB_HD bool operator()(int t, S& out) const { return fmt_csv_row(P, s, t, out); }
};

// Both passes of track s of the CSV text: 0 bytes for a masked track (fmt_stage_track).
template <bool WRITE>
EMB_HD uint32_t format_csv_track(const CsvParams& P, int64_t s, const ExpandLanes& L, char* stage) {
    if (P.mask && !P.mask[s]) return 0;
    bool ok = true;
    const uint32_t total = fmt_stage_track<WRITE>(FmtCsvItem{P, s}, P.T + 1, WRITE ? P.text + P.offsets[s] : nullptr, L, stage, ok);
    if (!ok) ll_flag(P.status, FMT_BAD_VALUE);
    return total;
}

}  // namespace emb
