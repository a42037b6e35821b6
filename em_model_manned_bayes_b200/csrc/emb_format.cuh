// emb_format.cuh -- the legacy text files of em_sample.m (initial.txt, transition.txt) formatted on the device: C's "%g" of a
// double and "%d" of an int64, and the per-track routines of k_format_{initial,transition}[_count] (emb_kernels.cu).
// __host__ __device__ like emb_events_expand.cuh, so that tests/emu runs the same code on the CPU.
//
// "%g" (C99 7.19.6.1, precision 6) is defined on the exact binary value v = m * 2^e: D = the 6-digit integer nearest to
// v / 10^k, ties to even, with k = X0 - 5 and X0 = floor(log10 |v|); a carry to 10^6 gives D = 10^5 and k + 1.  X = k + 5 is the
// exponent of the rounded value, "%f" style for -4 <= X < 6 and "%e" style otherwise, trailing zeros and a bare point dropped.
// The quotient and the comparison of the remainder with half the divisor are computed in exact integer arithmetic on
// A / B = v / 10^k (A = m 2^max(e,0) 10^max(-k,0), B = 2^max(-e,0) 10^max(k,0)): in 128 bits when A and B fit in 125 bits
// (every |v| from about 1e-17 to 1e37, so every sampled value and every id), otherwise in multi-word integers of up to 1280
// bits (subnormals need 10^329 * 2^53).  A double quotient only proposes q; the integer remainder corrects it.  Nothing is
// approximated, so the result is exact for every finite double (DESIGN.md section 13).
//
// Shape: one warp per track.  Lanes take consecutive items (transition: the rows of consecutive seconds; initial: the id and the
// values of the row); a warp scan of their byte lengths gives every lane its offset, the lanes move their items into the warp's
// shared-memory stage at those offsets, and the warp stores the stage as one contiguous block.  The count pass and the write pass
// emit through the same templates (fmt_emit_*, fmt_item) into a counting or a writing sink, so their byte counts agree by
// construction.
#pragma once
#include <cstdint>

#include "emb_events_expand.cuh"   // ExpandLanes (a warp on the device, one lane in the emulation), ll_flag

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

EMB_HD uint64_t fmt_bits(double v) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t b;
    std::memcpy(&b, &v, 8);
    return b;
#endif
}
EMB_HD int fmt_clz64(uint64_t x) {   // x != 0
#if defined(__CUDA_ARCH__)
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}
EMB_HD int fmt_ctz64(uint64_t x) {   // x != 0
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}

typedef unsigned __int128 u128;


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

// Multi-word unsigned integers for the quotients outside the 128-bit range (little-endian 32-bit limbs).
struct FmtBig {
    static constexpr int N = 40;   // 1280 bits: A <= 2^53 * 10^329 < 2^1147, B <= 2^1074
    uint32_t w[N];
    int n;                         // limbs in use; w[n-1] != 0 unless n == 0
};
EMB_HD void big_set(FmtBig& a, uint64_t v) {
    a.w[0] = (uint32_t)v;
    a.w[1] = (uint32_t)(v >> 32);
    a.n = a.w[1] ? 2 : a.w[0] ? 1 : 0;
}
EMB_HD void big_mul(FmtBig& a, uint32_t f) {
    if (!f) a.n = 0;
    uint64_t c = 0;
    for (int i = 0; i < a.n; ++i) {
        c += (uint64_t)a.w[i] * f;
        a.w[i] = (uint32_t)c;
        c >>= 32;
    }
    if (c) a.w[a.n++] = (uint32_t)c;
}
EMB_HD void big_mul_pow10(FmtBig& a, int j) {
    for (; j >= 9; j -= 9) big_mul(a, 1000000000u);
    uint32_t f = 1;
    for (; j > 0; --j) f *= 10u;
    if (f > 1) big_mul(a, f);
}
EMB_HD void big_shl(FmtBig& a, int s) {
    if (!a.n || !s) return;
    const int limbs = s >> 5, bits = s & 31;
    int n = a.n + limbs;
    a.w[n] = 0;
    for (int i = a.n - 1; i >= 0; --i) {
        const uint64_t x = (uint64_t)a.w[i] << bits;
        a.w[i + limbs + 1] |= (uint32_t)(x >> 32);
        a.w[i + limbs] = (uint32_t)x;
    }
    for (int i = 0; i < limbs; ++i) a.w[i] = 0;
    a.n = a.w[n] ? n + 1 : n;
}
EMB_HD int big_cmp(const FmtBig& a, const FmtBig& b) {
    if (a.n != b.n) return a.n < b.n ? -1 : 1;
    for (int i = a.n - 1; i >= 0; --i)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i] ? -1 : 1;
    return 0;
}
EMB_HD void big_sub(FmtBig& a, const FmtBig& b) {   // a -= b, a >= b
    int64_t c = 0;
    for (int i = 0; i < a.n; ++i) {
        c += (int64_t)a.w[i] - (i < b.n ? (int64_t)b.w[i] : 0);
        a.w[i] = (uint32_t)c;
        c >>= 32;
    }
    while (a.n && !a.w[a.n - 1]) --a.n;
}
EMB_HD void big_add(FmtBig& a, const FmtBig& b) {
    uint64_t c = 0;
    const int n = a.n > b.n ? a.n : b.n;
    for (int i = 0; i < n; ++i) {
        c += (uint64_t)(i < a.n ? a.w[i] : 0) + (i < b.n ? b.w[i] : 0);
        a.w[i] = (uint32_t)c;
        c >>= 32;
    }
    a.n = n;
    if (c) a.w[a.n++] = (uint32_t)c;
}
// a / 2^(32 (a.n - 3)) as a double (the top three limbs; relative error below 2^-63 before rounding)
EMB_HD double big_top(const FmtBig& a) {
    double r = 0.0;
    for (int i = a.n - 1; i >= 0 && i >= a.n - 3; --i) r = r * 4294967296.0 + (double)a.w[i];
    for (int i = a.n; i < 3; ++i) r *= 4294967296.0;   // fewer than three limbs: the same scale
    return r;
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

// Both passes of track s: the count pass returns its bytes; the write pass (WRITE) also stores them from P.offsets[s] on.
// stage: FMT_STAGE_BYTES of the warp's shared memory (write pass): a slot of FMT_ROW_MAX bytes per lane, into which the lane
// emits its item once, then the items packed at their scanned offsets, stored to global memory as one contiguous block.
template <bool TRANS, bool WRITE>
EMB_HD uint32_t format_track(const FormatParams& P, int64_t s, const ExpandLanes& L, char* stage) {
    const int W = ExpandLanes::width();
    const int items = TRANS ? P.T : P.n_initial + 1;
    const G6 id = TRANS ? fmt_g6((double)(P.first_id + s)) : G6{};
    char* dst = WRITE ? P.text + P.offsets[s] : nullptr;
    char* slot = stage + FMT_STAGE + L.lane * FMT_ROW_MAX;
    uint32_t total = 0;
    bool ok = true;
    for (int base = 0; base < items; base += W) {
        const int j = base + L.lane;
        int32_t len = 0;
        if (WRITE) {
            FmtWrite w{slot};
            if (j < items) fmt_item<TRANS>(P, s, j, id, w);
            len = (int32_t)(w.p - slot);
        } else {
            FmtCount c;
            if (j < items) ok &= fmt_item<TRANS>(P, s, j, id, c);
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
    if (!ok) ll_flag(P.status, FMT_BAD_VALUE);
    return total;
}

}  // namespace emb
