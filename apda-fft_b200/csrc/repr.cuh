// Shortest round-trip text of a double exactly as Python's float.__repr__ writes it (json.dumps uses it for floats and
// writes NaN / Infinity / -Infinity for the non-finite values).  Integer work only, exact for every double.
//
// Digits: Ryu (Ulf Adams, "Ryu: fast float-to-string conversion", PLDI 2018), the general 128-bit-table variant: the
// shortest decimal in the rounding interval of the double, the closest one to it when several are that short, ties to
// even.  This is what CPython's dtoa mode 0 returns.  The tables are generated from Python's exact integers by
// scripts/gen_present_tables.py.
// Layout (CPython's float_repr_style 'short', 'r' format with Py_DTSF_ADD_DOT_0): decpt = position of the decimal point
// relative to the first digit; fixed notation when -4 < decpt <= 16 (1e-4 <= |v| < 1e16) with ".0" on integral values,
// otherwise d[.ddd]e+XX / e-XX with at least two exponent digits.
#pragma once
#include <stdint.h>

#include "present_tables.cuh"

namespace repr {

__device__ __forceinline__ uint32_t pow5bits(uint32_t e) { return ((e * 1217359u) >> 19) + 1; }  // bitlen(5^e), e <= 3528
__device__ __forceinline__ uint32_t log10_pow2(uint32_t e) { return (e * 78913u) >> 18; }        // floor(e log10 2), e <= 1650
__device__ __forceinline__ uint32_t log10_pow5(uint32_t e) { return (e * 732923u) >> 20; }       // floor(e log10 5), e <= 2620

__device__ __forceinline__ uint32_t pow5_factor(uint64_t v) {  // v > 0
    uint32_t c = 0;
    for (;;) {
        const uint64_t q = v / 5;
        if (v - 5 * q != 0) return c;
        v = q;
        ++c;
    }
}
__device__ __forceinline__ bool multiple_of_pow5(uint64_t v, uint32_t p) { return pow5_factor(v) >= p; }
__device__ __forceinline__ bool multiple_of_pow2(uint64_t v, uint32_t p) { return (v & ((1ull << p) - 1)) == 0; }

// (m * mul) >> j for the 128-bit table entry mul = {lo, hi}, m < 2^55, 64 < j < 128
__device__ __forceinline__ uint64_t mul_shift(uint64_t m, const unsigned long long *mul, int32_t j) {
    const uint64_t lo = __ldg(mul), hi = __ldg(mul + 1);
    uint64_t high1 = __umul64hi(m, hi);
    const uint64_t low1 = m * hi;
    const uint64_t high0 = __umul64hi(m, lo);
    const uint64_t sum = high0 + low1;
    if (sum < high0) ++high1;
    const int dist = j - 64;
    return (high1 << (64 - dist)) | (sum >> dist);
}

struct Decimal {
    uint64_t digits;  // no trailing zero
    int32_t exp10;    // value = digits * 10^exp10
};

// shortest decimal of the positive finite double with biased exponent ie and mantissa field im (not both 0)
__device__ __forceinline__ Decimal shortest(uint64_t im, uint32_t ie) {
    int32_t e2;
    uint64_t m2;
    if (ie == 0) {
        e2 = 1 - 1023 - 52 - 2;
        m2 = im;
    } else {
        e2 = (int32_t)ie - 1023 - 52 - 2;
        m2 = (1ull << 52) | im;
    }
    const bool accept_bounds = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = im != 0 || ie <= 1;  // the lower neighbour is closer when m2 is a power of two

    uint64_t vr, vp, vm;
    int32_t e10;
    bool vm_zeros = false, vr_zeros = false;
    if (e2 >= 0) {
        const uint32_t q = log10_pow2((uint32_t)e2) - (e2 > 3);
        e10 = (int32_t)q;
        const int32_t k = APDA_POW5_INV_BITCOUNT + (int32_t)pow5bits(q) - 1;
        const int32_t i = -e2 + (int32_t)q + k;
        const unsigned long long *mul = kPow5InvSplit[q];
        vr = mul_shift(mv, mul, i);
        vp = mul_shift(mv + 2, mul, i);
        vm = mul_shift(mv - 1 - mm_shift, mul, i);
        if (q <= 21) {  // only one of mp, mv, mm can be a multiple of 5, if any
            if (mv % 5 == 0) vr_zeros = multiple_of_pow5(mv, q);
            else if (accept_bounds) vm_zeros = multiple_of_pow5(mv - 1 - mm_shift, q);
            else vp -= multiple_of_pow5(mv + 2, q);
        }
    } else {
        const uint32_t q = log10_pow5((uint32_t)-e2) - (-e2 > 1);
        e10 = (int32_t)q + e2;
        const int32_t i = -e2 - (int32_t)q;
        const int32_t k = (int32_t)pow5bits((uint32_t)i) - APDA_POW5_BITCOUNT;
        const int32_t j = (int32_t)q - k;
        const unsigned long long *mul = kPow5Split[i];
        vr = mul_shift(mv, mul, j);
        vp = mul_shift(mv + 2, mul, j);
        vm = mul_shift(mv - 1 - mm_shift, mul, j);
        if (q <= 1) {  // mv = 4 m2 has at least two trailing zero bits
            vr_zeros = true;
            if (accept_bounds) vm_zeros = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_zeros = multiple_of_pow2(mv, q);
        }
    }

    int32_t removed = 0;
    uint32_t last = 0;
    uint64_t out;
    if (vm_zeros || vr_zeros) {  // general case: an interval end or the value itself is exactly representable
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint64_t vr10 = vr / 10;
            vm_zeros &= vm - 10 * vm10 == 0;
            vr_zeros &= last == 0;
            last = (uint32_t)(vr - 10 * vr10);
            vr = vr10;
            vp = vp10;
            vm = vm10;
            ++removed;
        }
        if (vm_zeros) {
            for (;;) {
                const uint64_t vm10 = vm / 10;
                if (vm - 10 * vm10 != 0) break;
                const uint64_t vr10 = vr / 10;
                vr_zeros &= last == 0;
                last = (uint32_t)(vr - 10 * vr10);
                vr = vr10;
                vp = vp / 10;
                vm = vm10;
                ++removed;
            }
        }
        if (vr_zeros && last == 5 && vr % 2 == 0) last = 4;  // exactly ...50...0: round half to even
        out = vr + ((vr == vm && (!accept_bounds || !vm_zeros)) || last >= 5);
    } else {
        bool round_up = false;
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint64_t vr10 = vr / 10;
            round_up = vr - 10 * vr10 >= 5;
            vr = vr10;
            vp = vp10;
            vm = vm10;
            ++removed;
        }
        out = vr + (vr == vm || round_up);
    }
    Decimal d{out, e10 + removed};
    while (d.digits % 10 == 0) {  // rounding up can leave a trailing zero
        d.digits /= 10;
        ++d.exp10;
    }
    return d;
}

// the decimal digits of v < 10^20 as nibbles, least significant first (lo: digits 0..15, hi: 16..19); returns the count
__device__ __forceinline__ int bcd(uint64_t v, uint64_t &lo, uint32_t &hi) {
    int len = 1;
    for (uint64_t p = 10; len < 19 && v >= p; p *= 10) ++len;
    if (len == 19 && v >= 10000000000000000000ull) len = 20;
    lo = 0;
    hi = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        lo |= (v % 10) << (4 * i);
        v /= 10;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        hi |= (uint32_t)(v % 10) << (4 * i);
        v /= 10;
    }
    return len;
}
__device__ __forceinline__ char digit_at(uint64_t lo, uint32_t hi, int pos) {
    return (char)('0' + (pos < 16 ? (int)((lo >> (4 * pos)) & 15) : (int)((hi >> (4 * (pos - 16))) & 15)));
}

// Output sinks: Count only measures, Write stores the bytes.  Both run the same formatting code, so a row's measured
// length is the length it is written with.
struct Count {
    int64_t n = 0;
    __device__ __forceinline__ void put(char) { ++n; }
};
struct Write {
    char *p;
    int64_t n = 0;
    __device__ __forceinline__ void put(char c) { p[n++] = c; }
};

template <class O, int N>
__device__ __forceinline__ void put_lit(O &o, const char (&s)[N]) {
#pragma unroll
    for (int i = 0; i < N - 1; ++i) o.put(s[i]);
}

// str(v) of a Python int, 0 <= v < 2^63
template <class O>
__device__ __forceinline__ void put_int(O &o, uint64_t v) {
    uint64_t lo;
    uint32_t hi;
    const int len = bcd(v, lo, hi);
    for (int p = len - 1; p >= 0; --p) o.put(digit_at(lo, hi, p));
}

// repr(v) of a Python float; json.dumps' spelling of the non-finite values
template <class O>
__device__ __forceinline__ void put_double(O &o, double v) {
    const uint64_t b = (uint64_t)__double_as_longlong(v);
    const uint32_t ie = (uint32_t)(b >> 52) & 0x7ffu;
    const uint64_t im = b & ((1ull << 52) - 1);
    if (ie == 0x7ffu) {
        if (im) put_lit(o, "NaN");
        else if (b >> 63) put_lit(o, "-Infinity");
        else put_lit(o, "Infinity");
        return;
    }
    if (b >> 63) o.put('-');
    if (ie == 0 && im == 0) {
        put_lit(o, "0.0");
        return;
    }
    const Decimal d = shortest(im, ie);
    uint64_t lo;
    uint32_t hi;
    const int len = bcd(d.digits, lo, hi);
    const int decpt = d.exp10 + len;
    if (decpt <= -4 || decpt > 16) {
        o.put(digit_at(lo, hi, len - 1));
        if (len > 1) {
            o.put('.');
            for (int p = len - 2; p >= 0; --p) o.put(digit_at(lo, hi, p));
        }
        int x = decpt - 1;
        o.put('e');
        o.put(x < 0 ? '-' : '+');
        x = x < 0 ? -x : x;
        if (x >= 100) o.put((char)('0' + x / 100));
        o.put((char)('0' + x / 10 % 10));
        o.put((char)('0' + x % 10));
    } else if (decpt <= 0) {
        o.put('0');
        o.put('.');
        for (int i = 0; i < -decpt; ++i) o.put('0');
        for (int p = len - 1; p >= 0; --p) o.put(digit_at(lo, hi, p));
    } else if (decpt >= len) {
        for (int p = len - 1; p >= 0; --p) o.put(digit_at(lo, hi, p));
        for (int i = 0; i < decpt - len; ++i) o.put('0');
        o.put('.');
        o.put('0');
    } else {
        for (int p = len - 1; p >= 0; --p) {
            if (p == len - 1 - decpt) o.put('.');
            o.put(digit_at(lo, hi, p));
        }
    }
}

}  // namespace repr
