// Exact deposition sums: the fixed-point accumulator of a profile bin, its booking split and its conversion to a double.
//
// A floating-point atomicAdd into a bin rounds after every booking, and the order of the bookings at L2 changes from run to
// run, so the bins differ in their last bits. In exact-sum mode every booking v (a double: w dP, w P_dep or w, rounded once
// as in the float mode) is rounded to the quantum 2^-160 and added WITHOUT ERROR to integer words. Integer addition is
// associative, so the words do not depend on the order of the bookings, on which lane or SM made them, or on which device
// traced a ray (devices sum their words as integers). The profile is the correctly rounded double of the exact sum.
//
// Layout of one accumulator: TORJ_XS_WORDS = 8 signed 64-bit words; word k has weight 2^(28k - 160). A booking adds a signed
// 28-bit digit (|digit| < 2^28) to at most 3 consecutive words, with plain integer adds (RED on the device): a double's
// 53-bit significand spans at most 3 digits. Words are not kept normalised while bookings go in; carries are resolved only
// in the conversion.
//   - The quantum is fixed, not taken from a call's weights: only then is a plasma-set row bit-identical to the separate call
//     of that beam, and a shard's bookings identical to the same rays in the whole bundle. 2^-160 is far below any power a
//     trace books (a ray's shell power below 2^-161 of its weight contributes nothing); there are no subnormals.
//   - Value range: a booking must satisfy |v| < 2^64 (TORJ_XS_VMAX), so that its top digit falls into word 7. Others (and
//     NaN) are refused: counted in the refusal word and never added. The host refuses weights above TORJ_XS_WMAX, which
//     keeps w dP, w P_dep and w far inside that range.
//   - Headroom: a word changes by less than 2^28 per booking, so after at most TORJ_XS_MAX_BOOKINGS = 2^34 bookings into a
//     buffer |word| < 2^62, and a carry of the conversion (|carry| < 2^34 + 1) cannot overflow the next word. A buffer that
//     counts more bookings, or any refusal, is invalid: its conversion yields NaN and the results call fails.
// A buffer of n bins holds 2 status words (bookings made, bookings refused) followed by n * 8 words. Device buffers are
// summed over devices word by word, status words included, so the bound applies to the sum.
// Plain C++ (with __int128) and no CUDA dependency beyond the __host__ __device__ qualifier, so the host tests the same code
// (tests/test_exact_sum_format.py).
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define TORJ_XS_HD __host__ __device__ __forceinline__
#else
#define TORJ_XS_HD inline
#endif

#define TORJ_XS_WORDS 8                          // words per accumulator
#define TORJ_XS_DIGIT 28                         // bits per digit
#define TORJ_XS_Q 160                            // quantum 2^-TORJ_XS_Q
#define TORJ_XS_VMAX 18446744073709551616.0      // 2^64: |booking| must be below
#define TORJ_XS_WMAX 1099511627776.0             // 2^40: largest |weight| the host accepts in exact mode
#define TORJ_XS_MAX_BOOKINGS (1ll << 34)          // bookings a buffer may take (summed over devices)
#define TORJ_XS_STAT 2                           // status words before the bins: bookings, refusals

// int64 words of a buffer of n_bins accumulators with its status words
TORJ_XS_HD size_t torj_xs_buffer_words(size_t n_bins) { return n_bins * TORJ_XS_WORDS + TORJ_XS_STAT; }

struct TorjXsSplit {
    int ok;             // 0: refused (|v| >= 2^64 or NaN), nothing to add
    int k;              // first word, 0..TORJ_XS_WORDS-3
    long long d[3];     // digits for words k, k+1, k+2; |d| < 2^28, all of v's sign
};

// v rounded to the quantum (round half to even) as signed digits
TORJ_XS_HD TorjXsSplit torj_xs_split(double v) {
    TorjXsSplit r = {1, 0, {0, 0, 0}};
    if (!(fabs(v) < TORJ_XS_VMAX)) { r.ok = 0; return r; }
    uint64_t bits;
    memcpy(&bits, &v, sizeof bits);
    const int E = (int)((bits >> 52) & 0x7ff);
    uint64_t m = bits & ((1ull << 52) - 1);
    if (E) m |= 1ull << 52;
    if (!m) return r;
    const int s = (E ? E - 1075 : -1074) + TORJ_XS_Q;  // v = m 2^(s - 160)
    const uint64_t M = (1ull << TORJ_XS_DIGIT) - 1;
    if (s >= 0) {
        const int k = s / TORJ_XS_DIGIT, q = s % TORJ_XS_DIGIT;
        r.k = k;
        r.d[0] = (long long)((m << q) & M);
        r.d[1] = (long long)((m >> (TORJ_XS_DIGIT - q)) & M);
        r.d[2] = (long long)(m >> (2 * TORJ_XS_DIGIT - q));
        if (k > TORJ_XS_WORDS - 3) {  // |v| < 2^64: the digit past word 7 is 0
            r.k = TORJ_XS_WORDS - 3;
            r.d[2] = r.d[1]; r.d[1] = r.d[0]; r.d[0] = 0;
        }
    } else {
        const int t = -s;  // below the quantum: drop t bits, round half to even
        uint64_t q = 0;
        if (t <= 53) {
            q = m >> t;
            const uint64_t rem = m & ((1ull << t) - 1), half = 1ull << (t - 1);
            if (rem > half || (rem == half && (q & 1))) ++q;
        }
        r.d[0] = (long long)(q & M);
        r.d[1] = (long long)(q >> TORJ_XS_DIGIT);
    }
    if (v < 0) { r.d[0] = -r.d[0]; r.d[1] = -r.d[1]; r.d[2] = -r.d[2]; }
    return r;
}

// Host model of a booking (the device adds the same digits atomically)
TORJ_XS_HD void torj_xs_add(long long* w, TorjXsSplit s) {
    for (int j = 0; j < 3; ++j) w[s.k + j] += s.d[j];
}

// Carries: digits 0..6 into [0, 2^28), the rest into word 7 (value unchanged)
TORJ_XS_HD void torj_xs_normalize(long long* w) {
    for (int k = 0; k < TORJ_XS_WORDS - 1; ++k) {
        const long long c = w[k] >> TORJ_XS_DIGIT;  // floor division (arithmetic shift)
        w[k] -= c * (1ll << TORJ_XS_DIGIT);
        w[k + 1] += c;
    }
}

TORJ_XS_HD int torj_xs_bitlen(unsigned __int128 x) {
    int n = 0;
    while (x >> 64) { x >>= 64; n += 64; }
    uint64_t y = (uint64_t)x;
    while (y) { y >>= 1; ++n; }
    return n;
}

// The correctly rounded double (nearest, ties to even) of the exact value of words w[0..7] (not modified)
TORJ_XS_HD double torj_xs_to_double(const long long* w) {
    long long d[TORJ_XS_WORDS];
    for (int k = 0; k < TORJ_XS_WORDS; ++k) d[k] = w[k];
    torj_xs_normalize(d);
    const bool neg = d[TORJ_XS_WORDS - 1] < 0;
    if (neg) {  // magnitude: negate and normalise again (|word 7| < 2^62 leaves room)
        for (int k = 0; k < TORJ_XS_WORDS; ++k) d[k] = -d[k];
        torj_xs_normalize(d);
    }
    int t = TORJ_XS_WORDS - 1;
    while (t >= 0 && d[t] == 0) --t;
    if (t < 0) return 0.0;
    // the top digits into 128 bits (at least 101 of them when there are more digits), the rest into a sticky bit
    unsigned __int128 acc = (unsigned __int128)(uint64_t)d[t];
    int e = t * TORJ_XS_DIGIT;  // weight of acc's lowest bit, in quanta
    int k = t - 1;
    for (; k >= 0 && (acc >> 100) == 0; --k) {
        acc = (acc << TORJ_XS_DIGIT) | (uint64_t)d[k];
        e -= TORJ_XS_DIGIT;
    }
    bool sticky = false;
    for (; k >= 0; --k) sticky = sticky || d[k] != 0;
    const int L = torj_xs_bitlen(acc);
    uint64_t mant;
    if (L <= 53) {
        mant = (uint64_t)acc;  // exact (no dropped digit is nonzero: acc would have >= 101 bits)
    } else {
        const int sh = L - 53;
        mant = (uint64_t)(acc >> sh);
        const unsigned __int128 rem = acc & (((unsigned __int128)1 << sh) - 1), half = (unsigned __int128)1 << (sh - 1);
        if (rem > half || (rem == half && (sticky || (mant & 1)))) ++mant;  // 2^53 after a carry is still exact
        e += sh;
    }
    const double r = ldexp((double)mant, e - TORJ_XS_Q);
    return neg ? -r : r;
}

// Whether a buffer's status words (summed over devices) allow its conversion
TORJ_XS_HD bool torj_xs_valid(long long bookings, long long refused) {
    return refused == 0 && bookings >= 0 && bookings <= TORJ_XS_MAX_BOOKINGS;
}
