// emb_parse.cuh -- decimal text tables (the bodies of em_sample.m's initial.txt and transition.txt) parsed to fp64 on the device:
// the per-line routines of k_parse_lines and k_parse_values (emb_kernels.cu).  __host__ __device__ like emb_format.cuh, so that
// tests/emu runs the same code on the CPU.
//
// Lines and fields follow np.loadtxt: a line ends at '\n' or at the end of the text, fields are separated by runs of ' ', '\t' and
// '\r', a line without a field is skipped, every other line has exactly `cols` fields.  A field is
// [+-]?(d+(\.d*)?|\.d+)([eE][+-]?d+)? with at most 19 significant digits (leading and trailing zeros of the digit string do not
// count), so that its digits are an integer w < 10^19 < 2^64 and the field is (-1)^neg w 10^q.
//
// The value is the double nearest to w 10^q, ties to even (what Python's float() returns), decided exactly:
//  - w < 2^53 and |q| <= 22 (Clinger's fast path): w and 10^|q| are exact doubles, so one IEEE multiply or divide rounds
//    w 10^q correctly.  No multi-word integer is touched.
//  - otherwise a double proposed from w and powers of ten (a few ulps off at most) is settled against the exact decimal: the
//    candidate c moves up while w 10^q lies above the halfway point (c + c+)/2 = (2m+1) 2^(e-1) of c = m 2^e and its successor
//    c+, and down while it lies below the halfway point under c; a tie goes to the even significand.  The comparison is exact, in
//    the multi-word integers of emb_exact.cuh: w 10^max(q,0) 2^max(1-e,0) against (2m+1) 10^max(-q,0) 2^max(e-1,0).
// Range: with E = (significant digits) + q the decimal lies in [10^(E-1), 10^E).  E > 309 is above DBL_MAX and refused; E < -323
// lies below 10^-324, under half the smallest subnormal (2^-1075 > 2.4e-324), and gives +-0; so the settled tokens have
// q in [-342, 308].  The largest left side is 2^64 2^1075 = 2^1139 (a subnormal candidate, e - 1 = -1075), the largest right
// side (2^54) 10^342 < 2^1191; 38 limbs of 32 bits, within FmtBig's 40 (big_shl writes one limb past the result).  A candidate
// that moves past DBL_MAX (the decimal at or above DBL_MAX + ulp/2) is refused as out of range.
#pragma once
#include <cstdint>

#include "emb_exact.cuh"

namespace emb {

constexpr int PARSE_MAX_COLS = 256;
constexpr int PARSE_MAX_DIGITS = 19;
// error kinds: the error word is (1-based line << 2 | kind) and the smallest word wins (the first line, then the lowest kind)
constexpr int PARSE_E_TOKEN = 0;    // a field that is not a decimal number
constexpr int PARSE_E_DIGITS = 1;   // more than 19 significant digits
constexpr int PARSE_E_RANGE = 2;    // rounds to +-inf
constexpr int PARSE_E_FIELDS = 3;   // a line with fields, but not `cols` of them
constexpr unsigned long long PARSE_NO_ERROR = ~0ull;

struct ParseParams {
    const char* text;
    int64_t bytes;
    int32_t cols;
    int32_t aligned;                  // text is 16-byte aligned (vector loads in line discovery)
    int64_t chunks;                   // PARSE_CHUNK-byte chunks of the text
    uint32_t* chunk_newlines;         // [chunks] (k_parse_newline_count)
    const long long* newlines_before; // [chunks + 1] exclusive scan of chunk_newlines
    int64_t lines;                    // newlines + 1 (the last line may be empty)
    long long* starts;                // [lines + 1]: line i is [starts[i], starts[i+1] - 1); starts[lines] = bytes + 1
    uint32_t* rows;                   // [lines] 1 for a line with fields, 0 for a blank line (k_parse_lines)
    const long long* row_of;          // [lines + 1] exclusive scan of rows (k_parse_values)
    double* values;                   // [rows][cols]
    unsigned long long* error;        // PARSE_NO_ERROR or the first error word
};

EMB_HD bool parse_sep(char c) { return c == ' ' || c == '\t' || c == '\r'; }
EMB_HD bool parse_digit(char c) { return c >= '0' && c <= '9'; }

// a token as (-1)^neg w 10^q, w without leading or trailing zeros (or 0); sig = digits of w
struct ParseDec {
    uint64_t w;
    int64_t q;
    int32_t sig;
    bool neg;
};

// [p, e) is one token (no separator inside); 0 or -1 - PARSE_E_*
EMB_HD int parse_token(const char* p, const char* e, ParseDec& d) {
    d.w = 0;
    d.q = 0;
    d.sig = 0;
    d.neg = false;
    if (*p == '+' || *p == '-') d.neg = *p++ == '-';
    int64_t pend = 0;   // zeros after the last nonzero digit, not yet in w
    int digits = 0;
    bool frac = false;
    for (; p < e; ++p) {
        const char c = *p;
        if (c == '.') {
            if (frac) break;
            frac = true;
            continue;
        }
        if (!parse_digit(c)) break;
        ++digits;
        if (frac) --d.q;
        if (c == '0') {
            if (d.sig) ++pend;
            continue;
        }
        if (d.sig + pend + 1 > PARSE_MAX_DIGITS) return -1 - PARSE_E_DIGITS;
        d.sig += (int32_t)pend + 1;   // the pending zeros and this digit
        for (; pend > 0; --pend) d.w *= 10u;
        d.w = d.w * 10u + (uint64_t)(c - '0');
    }
    if (!digits) return -1 - PARSE_E_TOKEN;
    d.q += pend;
    if (p < e && (*p == 'e' || *p == 'E')) {
        ++p;
        bool eneg = false;
        if (p < e && (*p == '+' || *p == '-')) eneg = *p++ == '-';
        if (p == e) return -1 - PARSE_E_TOKEN;
        int64_t x = 0;
        for (; p < e && parse_digit(*p); ++p)
            if (x < 100000000) x = x * 10 + (*p - '0');   // saturates far outside the range of a double
        if (p < e) return -1 - PARSE_E_TOKEN;
        d.q += eneg ? -x : x;
    }
    return p == e ? 0 : -1 - PARSE_E_TOKEN;
}

EMB_HD double parse_from_bits(uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)b);
#else
    double v;
    std::memcpy(&v, &b, 8);
    return v;
#endif
}

// 10^k for 0 <= k <= 22, exact (every factor and product is a power of ten below 2^76 with at most 53 significant bits)
EMB_HD double parse_pow10_exact(int k) {
    double r = 1.0, b = 10.0;
    for (; k; k >>= 1, b *= b)
        if (k & 1) r *= b;
    return r;
}
// about 10^k for 0 <= k < 512 from correctly rounded factors (a few ulps: only the proposal of the exact path uses it)
EMB_HD double parse_pow10_approx(int k) {
    double r = parse_pow10_exact(k & 15);
    if (k & 16) r *= 1e16;
    if (k & 32) r *= 1e32;
    if (k & 64) r *= 1e64;
    if (k & 128) r *= 1e128;
    if (k & 256) r *= 1e256;
    return r;
}

// sign of w 10^q - (c + c+) / 2 for the positive double (or zero) with bits c: the halfway point is (2m+1) 2^(e-1)
EMB_HD int parse_cmp_mid(uint64_t w, int q, uint64_t c) {
    const int be = (int)(c >> 52);
    const uint64_t m = (c & 0xFFFFFFFFFFFFFull) | (be ? 1ull << 52 : 0ull);
    const int e1 = (be ? be : 1) - 1075 - 1;
    FmtBig A, B;
    big_set(A, w);
    big_set(B, 2 * m + 1);
    if (q > 0) big_mul_pow10(A, q);
    else big_mul_pow10(B, -q);
    if (e1 > 0) big_shl(B, e1);
    else big_shl(A, -e1);
    return big_cmp(A, B);
}

// |value| of w 10^q, w != 0, -342 <= q <= 308, outside the fast path; `inf` if it rounds to infinity
EMB_HD double parse_settle(uint64_t w, int q, bool& inf) {
    double x = (double)w;
    if (q >= 0) x *= parse_pow10_approx(q);
    else if (q >= -300) x /= parse_pow10_approx(-q);
    else x = x / parse_pow10_approx(-q - 300) / 1e300;
    constexpr uint64_t DBL_MAX_BITS = 0x7FEFFFFFFFFFFFFFull;
    uint64_t c = fmt_bits(x) & ~(1ull << 63);
    if (c > DBL_MAX_BITS) c = DBL_MAX_BITS;
    for (;;) {
        const int up = parse_cmp_mid(w, q, c);
        if (up > 0 || (up == 0 && (c & 1u))) {   // nearer to c+, or a tie and c's significand odd
            if (c == DBL_MAX_BITS) {
                inf = true;
                return 0.0;
            }
            ++c;
            continue;
        }
        if (c) {
            const int down = parse_cmp_mid(w, q, c - 1);
            if (down < 0 || (down == 0 && !((c - 1) & 1u))) {   // nearer to c-, or a tie and c-'s significand even
                --c;
                continue;
            }
        }
        return parse_from_bits(c);
    }
}

// the double of a token (sign included); `range` if it rounds to +-inf
EMB_HD double parse_value(const ParseDec& d, bool& range) {
    double v = 0.0;
    range = false;
    if (d.w) {
        const int64_t E = d.sig + d.q;
        if (E > 309) {
            range = true;
        } else if (E >= -323) {
            const int q = (int)d.q;
            if (d.w < (1ull << 53) && q >= -22 && q <= 22) v = q >= 0 ? (double)d.w * parse_pow10_exact(q) : (double)d.w / parse_pow10_exact(-q);
            else v = parse_settle(d.w, q, range);
        }
    }
    return d.neg ? -v : v;
}

// One line [p, e): the number of fields (0 for a blank line), or -1 - PARSE_E_*.  VALUES: the values to out[0 .. cols).
// Without VALUES a token is only checked, and its value computed only where it could round to infinity (E >= 309).
template <bool VALUES>
EMB_HD int parse_line(const char* p, const char* e, int cols, double* out) {
    int f = 0;
    while (true) {
        while (p < e && parse_sep(*p)) ++p;
        if (p == e) break;
        const char* t = p;
        while (p < e && !parse_sep(*p)) ++p;
        if (f == cols) return -1 - PARSE_E_FIELDS;
        ParseDec d;
        const int rc = parse_token(t, p, d);
        if (rc) return rc;
        bool range = false;
        if (VALUES) out[f] = parse_value(d, range);
        else if (d.w && d.sig + d.q >= 309) parse_value(d, range);
        if (range) return -1 - PARSE_E_RANGE;
        ++f;
    }
    return f == 0 || f == cols ? f : -1 - PARSE_E_FIELDS;
}

EMB_HD void parse_error(unsigned long long* word, int64_t line, int kind) {
    const unsigned long long v = ((unsigned long long)(line + 1) << 2) | (unsigned long long)kind;
#if defined(__CUDA_ARCH__)
    atomicMin(word, v);
#else
    if (v < *word) *word = v;
#endif
}

// line i of the text (emb_kernels.cu: k_parse_lines): P.rows[i], or the error word
EMB_HD void parse_check_line(const ParseParams& P, int64_t i) {
    const char* p = P.text + P.starts[i];
    const char* e = P.text + (P.starts[i + 1] - 1);
    const int f = parse_line<false>(p, e, P.cols, nullptr);
    if (f < 0) parse_error(P.error, i, -1 - f);
    P.rows[i] = f > 0 ? 1u : 0u;
}

// line i (emb_kernels.cu: k_parse_values): its values to row P.row_of[i], if it is a row
EMB_HD void parse_values_line(const ParseParams& P, int64_t i) {
    const long long r = P.row_of[i];
    if (P.row_of[i + 1] == r) return;
    parse_line<true>(P.text + P.starts[i], P.text + (P.starts[i + 1] - 1), P.cols, P.values + r * P.cols);
}

}  // namespace emb
