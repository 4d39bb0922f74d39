/*
 * ste_text.cuh - exact "%.18e" conversion of doubles, the format np.savetxt writes by default (CPython's
 * PyOS_double_to_string(x, 'e', 18): Gay's dtoa mode 2, 19 significant digits, correctly rounded, ties to even).
 *
 * Method.  A finite x != 0 is m * 2^e (m < 2^53).  Its output is the 19-digit integer D = round(x * 10^(18 - k)) with
 * 10^18 <= x * 10^(18 - k) < 10^19, i.e. k = floor(log10 x), and "d.ddd...e+k".  D is first estimated in double-double
 * arithmetic: m * 10^r (r = s mod 16, 10^r exact) is an exact product, times 10^(16 j) from a 41-entry table rounded to
 * 106 bits, scaled by 2^(e + exponent of the entry).  The estimate's relative error is below 2^-102, so its absolute
 * error is below 2^-36 for the values of D that occur (< 2^66).  The estimate decides k and the rounding of D unless
 * it lies within kEps = 2^-24 of a decision boundary: 10^18 or 10^19 (is x below 10^k, or at least 10^(k+1)?), or a
 * half-integer (does x * 10^s lie below, above or exactly on q + 1/2?).  Those cases - exact powers of ten, exact ties
 * such as m * 2^-5 with 20 significant digits, and a fraction of about 2^-23 of all other values - are decided exactly
 * (exact powers 10^0 .. 10^22, doubles themselves, by comparing doubles; the rest as follows):
 * both sides are written as integers times powers of 2 and 5, the power of 5 is multiplied out into a big integer of
 * 32-bit limbs (at most 862 bits: 5^343 times a 65-bit integer) and the two sides are compared bit by bit.
 *
 * The functions are __host__ __device__ so that the same code can be checked on the CPU.
 */
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define STE_TEXT_HD __host__ __device__ __forceinline__
#define STE_TEXT_HD_NOINLINE __host__ __device__ __noinline__
#else
#define STE_TEXT_HD inline
#define STE_TEXT_HD_NOINLINE
#endif

namespace ste {
namespace text {

typedef unsigned __int128 u128;

// Longest field: "-1.234567890123456789e-308" (26 bytes), plus its separator.
constexpr int kMaxField = 26;
constexpr int kMaxValueBytes = kMaxField + 1;

// meta word of a converted value: kind (bits 0-1), sign (bit 2), newline after the value (bit 3), k + 512 (bits 8-19)
constexpr int kKindFinite = 0, kKindInf = 1, kKindNan = 2;
constexpr int32_t kMetaNeg = 0x4, kMetaNewline = 0x8;

constexpr uint64_t kP18 = 1000000000000000000ull, kP19 = 10000000000000000000ull;

struct Pow10Entry {
    double hi, lo;   // 10^(16 j) = (hi + lo) * 2^e2, 1 <= hi < 2, hi + lo rounded to 106 bits
    int e2;
};

// 10^(16 j) for j = -19 .. 21 (s = 18 - k spans -291 .. 343).  Generated with Python's fractions.Fraction:
// hi = float(f), lo = float(f - hi) with f = 10^(16 j) / 2^e2 in [1, 2).
#define STE_TEXT_POW10_BY16 {                                                                                    \
    {0x1.18e3b9b374169p+0, 0x1.259ff0c08b7f2p-55, -1010},   /* 1e-304 */                                          \
    {0x1.37d99cc506d59p+0, -0x1.44588e4c035e8p-54, -957},   /* 1e-288 */                                          \
    {0x1.5a391d56bdc87p+0, 0x1.b36d1921b2800p-54, -904},   /* 1e-272 */                                           \
    {0x1.8062864ac6f43p+0, 0x1.39fa911155ff0p-55, -851},   /* 1e-256 */                                           \
    {0x1.aac0bf9b9e65cp+0, 0x1.d6fb1e4a9a909p-55, -798},   /* 1e-240 */                                           \
    {0x1.d9ca79d89462ap+0, -0x1.425b0740a9caep-55, -745},   /* 1e-224 */                                          \
    {0x1.0701bd527b498p+0, -0x1.cfdedc1a30d30p-54, -691},   /* 1e-208 */                                          \
    {0x1.23ff06eea847ap+0, -0x1.fcc24e7cae5cfp-54, -638},   /* 1e-192 */                                          \
    {0x1.442e4fb671960p+0, 0x1.7dc56d0072d28p-58, -585},   /* 1e-176 */                                           \
    {0x1.67e9c127b6e74p+0, 0x1.26b3da42cecadp-56, -532},   /* 1e-160 */                                           \
    {0x1.8f9574dcf8a70p+0, 0x1.647f32529774bp-54, -479},   /* 1e-144 */                                           \
    {0x1.bba08cf8c979dp+0, -0x1.afa9c1a60497dp-54, -426},   /* 1e-128 */                                          \
    {0x1.ec866b79e0cbap+0, 0x1.bea6a30bdaffap-54, -373},   /* 1e-112 */                                           \
    {0x1.116805effaeaap+0, 0x1.cd88ede5810c7p-54, -319},   /* 1e-96 */                                            \
    {0x1.2f8ac174d6123p+0, 0x1.a5dccd879fc96p-55, -266},   /* 1e-80 */                                            \
    {0x1.50ffd44f4a73dp+0, 0x1.a53f2398d747bp-55, -213},   /* 1e-64 */                                            \
    {0x1.7624f8a762fd8p+0, 0x1.595560c018581p-55, -160},   /* 1e-48 */                                            \
    {0x1.9f623d5a8a733p+0, -0x1.a2cc10f3892d4p-54, -107},   /* 1e-32 */                                           \
    {0x1.cd2b297d889bcp+0, 0x1.5b4c2ebe68799p-55, -54},   /* 1e-16 */                                             \
    {0x1.0000000000000p+0, 0x0.0p+0, 0},   /* 1e0 */                                                              \
    {0x1.1c37937e08000p+0, 0x0.0p+0, 53},   /* 1e16 */                                                            \
    {0x1.3b8b5b5056e17p+0, -0x1.3107f00000000p-54, 106},   /* 1e32 */                                             \
    {0x1.5e531a0a1c873p+0, -0x1.14b4c7a76a406p-54, 159},   /* 1e48 */                                             \
    {0x1.84f03e93ff9f5p+0, -0x1.2ac340948e389p-55, 212},   /* 1e64 */                                             \
    {0x1.afcef51f0fb5fp+0, -0x1.08f322e84da10p-61, 265},   /* 1e80 */                                             \
    {0x1.df67562d8b363p+0, -0x1.ae9d180b58861p-54, 318},   /* 1e96 */                                             \
    {0x1.0a1f5b8132466p+0, 0x1.4f01f167b5e30p-54, 372},   /* 1e112 */                                             \
    {0x1.27748f9301d32p+0, -0x1.901cc86649e4ap-54, 425},   /* 1e128 */                                            \
    {0x1.4805738b51a75p+0, -0x1.18a0e9df9363ap-55, 478},   /* 1e144 */                                            \
    {0x1.6c2d4256ffcc3p+0, -0x1.56a2119e533adp-57, 531},   /* 1e160 */                                            \
    {0x1.945145230b378p+0, -0x1.b20a11c22bf0cp-57, 584},   /* 1e176 */                                            \
    {0x1.c0e1ef1a724ebp+0, -0x1.4abd220ed605cp-54, 637},   /* 1e192 */                                            \
    {0x1.f25c186a6f04cp+0, 0x1.45a7709a56ccep-55, 690},   /* 1e208 */                                             \
    {0x1.14a52dffc6799p+0, 0x1.2f82bd6b70d9ap-55, 744},   /* 1e224 */                                             \
    {0x1.33234de7ad7e3p+0, -0x1.34a66b24bc3ebp-56, 797},   /* 1e240 */                                            \
    {0x1.54fdd7f73bf3cp+0, -0x1.7222446fe4670p-55, 850},   /* 1e256 */                                            \
    {0x1.7a93a2954f3b8p+0, -0x1.beda693cdd93bp-54, 903},   /* 1e272 */                                            \
    {0x1.a44df832b8d46p+0, -0x1.ce31f3444e400p-57, 956},   /* 1e288 */                                            \
    {0x1.d2a1be4048f90p+0, 0x1.fea3e35c17799p-54, 1009},   /* 1e304 */                                            \
    {0x1.03085e53e599cp+0, 0x1.baf3508ac1807p-54, 1063},   /* 1e320 */                                            \
    {0x1.1f9584aeab1ddp+0, -0x1.8cef62d87aad1p-54, 1116},   /* 1e336 */                                           \
}

// 10^0 .. 10^22: every one is exactly a double (5^22 < 2^53)
#define STE_TEXT_POW10_SMALL {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, \
                              1e18, 1e19, 1e20, 1e21, 1e22}

#ifdef __CUDACC__
__device__ const Pow10Entry kPow10By16Dev[41] = STE_TEXT_POW10_BY16;
__device__ const double kPow10SmallDev[23] = STE_TEXT_POW10_SMALL;
#endif
static const Pow10Entry kPow10By16Host[41] = STE_TEXT_POW10_BY16;
static const double kPow10SmallHost[23] = STE_TEXT_POW10_SMALL;

STE_TEXT_HD Pow10Entry pow10_by16(int j) {
#ifdef __CUDA_ARCH__
    return kPow10By16Dev[j + 19];
#else
    return kPow10By16Host[j + 19];
#endif
}

STE_TEXT_HD double pow10_small(int r) {
#ifdef __CUDA_ARCH__
    return kPow10SmallDev[r];
#else
    return kPow10SmallHost[r];
#endif
}

// ---- exact comparison: big integers of 32-bit limbs ------------------------------------------------------------ //
constexpr int kLimbs = 28;   // 896 bits >= 65 + ceil(343 * log2 5) = 862

struct Big {
    uint32_t w[kLimbs];
    int n;   // limbs in use; w[n-1] != 0 unless n == 0
};

STE_TEXT_HD void big_set(Big &b, u128 v) {
    b.n = 0;
    while (v) { b.w[b.n++] = (uint32_t)v; v >>= 32; }
}

STE_TEXT_HD void big_mul_small(Big &b, uint32_t f) {
    uint64_t carry = 0;
    for (int i = 0; i < b.n; ++i) {
        const uint64_t t = (uint64_t)b.w[i] * f + carry;
        b.w[i] = (uint32_t)t;
        carry = t >> 32;
    }
    if (carry) b.w[b.n++] = (uint32_t)carry;
}

STE_TEXT_HD void big_mul_pow5(Big &b, int p) {
    for (; p >= 13; p -= 13) big_mul_small(b, 1220703125u);   // 5^13 < 2^32
    uint32_t f = 1;
    for (; p > 0; --p) f *= 5;
    if (f != 1) big_mul_small(b, f);
}

STE_TEXT_HD int bitlen128(u128 v) {
    int n = 0;
    while (v) { ++n; v >>= 1; }
    return n;
}

STE_TEXT_HD int big_bitlen(const Big &b) {
    if (b.n == 0) return 0;
    uint32_t top = b.w[b.n - 1];
    int n = 32 * (b.n - 1);
    while (top) { ++n; top >>= 1; }
    return n;
}

// bits [lo, lo + 128) of b
STE_TEXT_HD u128 big_bits(const Big &b, int lo) {
    u128 r = 0;
    for (int i = 127; i >= 0; --i) {
        const int bit = lo + i, limb = bit >> 5;
        r = (r << 1) | (limb < b.n ? (b.w[limb] >> (bit & 31)) & 1u : 0u);
    }
    return r;
}

// any of the bits [0, nbits) of b set
STE_TEXT_HD bool big_low_nonzero(const Big &b, int nbits) {
    for (int i = 0; i < b.n && 32 * i < nbits; ++i) {
        const int keep = nbits - 32 * i;
        const uint32_t mask = keep >= 32 ? 0xffffffffu : ((1u << keep) - 1u);
        if (b.w[i] & mask) return true;
    }
    return false;
}

// sign of X * 2^w - Y, X > 0, Y > 0
STE_TEXT_HD int big_cmp_shifted(const Big &X, int w, u128 Y) {
    const int nx = big_bitlen(X) + w, ny = bitlen128(Y);
    if (nx != ny) return nx > ny ? 1 : -1;
    // nx == ny <= 128: the integer part of X * 2^w has ny bits
    const u128 top = w >= 0 ? (big_bits(X, 0) << w) : big_bits(X, -w);
    if (top != Y) return top > Y ? 1 : -1;
    return (w < 0 && big_low_nonzero(X, -w)) ? 1 : 0;
}

// sign of A * 2^a2 * 5^a5 - B * 2^b2 * 5^b5 (A, B > 0), exactly
STE_TEXT_HD_NOINLINE int cmp_exact(u128 A, int a2, int a5, u128 B, int b2, int b5) {
    Big X;
    const int p2 = a2 - b2, p5 = a5 - b5;
    if (p5 >= 0) {   // A * 5^p5 * 2^p2 vs B
        big_set(X, A);
        big_mul_pow5(X, p5);
        return big_cmp_shifted(X, p2, B);
    }
    big_set(X, B);   // A * 2^p2 vs B * 5^-p5  <=>  -(X * 2^-p2 - A)
    big_mul_pow5(X, -p5);
    return -big_cmp_shifted(X, -p2, A);
}

// sign of x - 10^k for x = m * 2^e = ax.  For 0 <= k <= 22, 10^k is a double, so comparing the doubles is exact; this
// decides the exact powers of ten the CLI's files are full of (1.0 prior variances, 1-hour steps) without big integers.
STE_TEXT_HD int cmp_pow10(uint64_t m, int e, double ax, int k) {
    if (k >= 0 && k <= 22) {
        const double p = pow10_small(k);
        return ax < p ? -1 : (ax > p ? 1 : 0);
    }
    return cmp_exact(m, e, 0, 1, k, k);
}

// ---- the conversion ---------------------------------------------------------------------------------------------- //
constexpr double kEps = 1.0 / 16777216.0;   // 2^-24, far above the estimate's error (< 2^-36)

// q + f (q integer, 0 <= f < 1) estimates x * 10^(18 - k) for x = m * 2^e.  Returns -1 when the estimate is far below
// 2^59 (k too large), +1 when it is 2^64 or more (k too small), else 0.
STE_TEXT_HD int estimate(uint64_t m, int e, int k, uint64_t &q, double &f) {
    const int s = 18 - k;
    const int j = (s >= 0) ? s / 16 : -((15 - s) / 16);
    const int r = s - 16 * j;
    const Pow10Entry t = pow10_by16(j);
    const double md = (double)m, pr = pow10_small(r);
    const double ph = md * pr, pl = fma(md, pr, -ph);   // exact: m * 10^r = ph + pl
    const double h = ph * t.hi, hl = fma(ph, t.hi, -h);
    const double l = hl + (ph * t.lo + pl * t.hi);
    double dh = h + l;
    double dl = l - (dh - h);
    dh = ldexp(dh, e + t.e2);
    dl = ldexp(dl, e + t.e2);
    if (!(dh < 18446744073709551616.0)) return 1;
    if (dh < 576460752303423488.0) return -1;   // 2^59 < 10^18
    const double fl = floor(dl);
    q = (uint64_t)dh + (uint64_t)(int64_t)fl;
    f = dl - fl;
    return 0;
}

// x finite and != 0, |x| = m * 2^e: the 19 digits D and decimal exponent k of "%.18e"
STE_TEXT_HD void decimal19(uint64_t m, int e, double ax, uint64_t &digits, int &k_out) {
    int k = (int)floor(log10(ax));
    uint64_t q = 0;
    double f = 0.0;
    for (int it = 0; it < 8; ++it) {
        const int far = estimate(m, e, k, q, f);
        bool below = far < 0, above = far > 0;
        if (!far) {
            if (q < kP18 - 1 || (q == kP18 - 1 && f <= 1.0 - kEps)) below = true;
            else if ((q == kP18 - 1) || (q == kP18 && f < kEps)) below = cmp_pow10(m, e, ax, k) < 0;          // x < 10^k ?
            else if (q > kP19 || (q == kP19 && f >= kEps)) above = true;
            else if ((q == kP19 - 1 && f > 1.0 - kEps) || q == kP19) above = cmp_pow10(m, e, ax, k + 1) >= 0;
        }
        if (below) --k;
        else if (above) ++k;
        else break;
    }
    const int s = 18 - k;
    uint64_t d = q;
    if (f > 0.5 + kEps) {
        d = q + 1;
    } else if (f >= 0.5 - kEps) {   // x * 10^s against q + 1/2: m * 2^(e+1+s) * 5^s against 2q + 1
        const int c = cmp_exact(m, e + 1 + s, s, (u128)q * 2u + 1u, 0, 0);
        d = (c > 0 || (c == 0 && (q & 1u))) ? q + 1 : q;
    }
    if (d == kP19) {   // rounding carried into the next power of ten
        d = kP18;
        ++k;
    }
    digits = d;
    k_out = k;
}

// Converts x: digits (0 for zero, inf, nan) and the meta word (without kMetaNewline).
STE_TEXT_HD void convert(double x, uint64_t &digits, int32_t &meta) {
    uint64_t bits;
    memcpy(&bits, &x, 8);
    const bool neg = (bits >> 63) != 0;
    const int biased = (int)((bits >> 52) & 0x7ff);
    const uint64_t frac = bits & ((1ull << 52) - 1);
    digits = 0;
    if (biased == 0x7ff) {
        meta = frac ? kKindNan : (kKindInf | (neg ? kMetaNeg : 0));   // CPython prints every NaN as "nan"
        return;
    }
    int k = 0;
    if (biased != 0 || frac != 0) {
        const uint64_t m = biased ? (frac | (1ull << 52)) : frac;
        const int e = biased ? biased - 1075 : -1074;
        decimal19(m, e, fabs(x), digits, k);
    }
    meta = kKindFinite | (neg ? kMetaNeg : 0) | ((k + 512) << 8);
}

// Field length (without separator) of a converted value.
STE_TEXT_HD int field_length(int32_t meta) {
    const int neg = (meta & kMetaNeg) ? 1 : 0;
    switch (meta & 3) {
    case kKindInf: return 3 + neg;
    case kKindNan: return 3;
    default: {
        const int k = ((meta >> 8) & 0xfff) - 512;
        return neg + 22 + ((k >= 100 || k <= -100) ? 3 : 2);   // d.<18 digits>e<sign><2 or 3 digits>
    }
    }
}

// Writes the field of a converted value followed by its separator (' ' or '\n'); returns the bytes written.
STE_TEXT_HD int format_field(uint64_t digits, int32_t meta, char *out) {
    int p = 0;
    if (meta & kMetaNeg) out[p++] = '-';
    const int kind = meta & 3;
    if (kind == kKindInf || kind == kKindNan) {
        const char *w = kind == kKindInf ? "inf" : "nan";
        out[p++] = w[0]; out[p++] = w[1]; out[p++] = w[2];
    } else {
        for (int i = 19; i >= 2; --i) {   // out[p + 2 .. p + 19] = digits 2 .. 19, out[p] = leading digit
            out[p + i] = (char)('0' + digits % 10);
            digits /= 10;
        }
        out[p] = (char)('0' + digits);
        out[p + 1] = '.';
        p += 20;
        int k = ((meta >> 8) & 0xfff) - 512;
        out[p++] = 'e';
        out[p++] = k < 0 ? '-' : '+';
        if (k < 0) k = -k;
        if (k >= 100) { out[p++] = (char)('0' + k / 100); k %= 100; }
        out[p++] = (char)('0' + k / 10);
        out[p++] = (char)('0' + k % 10);
    }
    out[p++] = (meta & kMetaNewline) ? '\n' : ' ';
    return p;
}

}  // namespace text
}  // namespace ste
