// emb_exact.cuh -- exact integer arithmetic shared by the text formatter (emb_format.cuh) and the text parser (emb_parse.cuh):
// the bits of a double, and multi-word unsigned integers for the decisions that do not fit in 128 bits.
// __host__ __device__ so that tests/emu runs the same code on the CPU.
#pragma once
#include <cstdint>
#include <cstring>

#include "emb_device.cuh"   // EMB_HD

namespace emb {

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

// Multi-word unsigned integers for the quotients outside the 128-bit range (little-endian 32-bit limbs).
struct FmtBig {
    static constexpr int N = 40;   // 1280 bits; the bounds of each user are derived in emb_format.cuh and emb_parse.cuh
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

}  // namespace emb
