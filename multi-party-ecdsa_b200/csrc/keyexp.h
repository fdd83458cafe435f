// Sliding windows over key exponents, and the slot orders that make them warp-uniform.
//
// The exponents of a key row (N, p, q, p-1, q-1, q mod (p-1), p mod (q-1)) are constants of the row.  Left-to-right sliding
// windows of width KEYEXP_BITS over odd digits need fewer products than the 5-bit fixed windows of per-unit exponents, but
// the schedule (where the products fall) depends on the exponent.  The job kernels run it only on classes whose instances
// are ordered by key row (keyexp_order), so every lane group of a warp holds the same exponent and follows the same
// schedule; the warp walks the windows of its first lane group's exponent.
//
// Plain C++ with host/device qualifiers: the job kernels and the CPU tests (tests/test_keyexp_schedule.py) share it.
#pragma once
#include <cstddef>
#include <cstdint>

#ifdef __CUDACC__
#define KEYEXP_HD __host__ __device__ __forceinline__
#else
#define KEYEXP_HD inline
#endif

namespace tecdsa {

static constexpr int KEYEXP_BITS = 6;                          // width 7 needs the same products and twice the table
static constexpr int KEYEXP_TBL = 1 << (KEYEXP_BITS - 1);      // odd powers x, x^3, .., x^(2^KEYEXP_BITS - 1)
static constexpr uint32_t ORDER_PAD = 0x80000000u;             // flag of a padding slot; its low bits name the run's first unit

KEYEXP_HD int keyexp_clz(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __clz(x);
#else
    return x ? __builtin_clz(x) : 32;
#endif
}
KEYEXP_HD int keyexp_ctz(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __ffs(x) - 1;
#else
    return __builtin_ctz(x);
#endif
}

// highest set bit of the little-endian limb array `e` at or below bit `from`; -1 if there is none
KEYEXP_HD int keyexp_top(const uint32_t* e, int from) {
    while (from >= 0) {
        const uint32_t w = e[from >> 5] & (0xffffffffu >> (31 - (from & 31)));
        if (w) return (from & ~31) + 31 - keyexp_clz(w);
        from = (from & ~31) - 1;
    }
    return -1;
}

// The window whose top bit is the set bit `top`: its odd digit (bits lo..top) and its low bit lo.  The next window starts at
// keyexp_top(e, lo - 1), so windows start at least KEYEXP_BITS bits apart: at most ceil(bits / KEYEXP_BITS) of them.
KEYEXP_HD int keyexp_window(const uint32_t* e, int top, uint32_t& digit) {
    const int lo = top >= KEYEXP_BITS - 1 ? top - (KEYEXP_BITS - 1) : 0;
    const int limb = lo >> 5;
    const uint64_t hi = (top >> 5) > limb ? (uint64_t)e[limb + 1] << 32 : 0;
    uint32_t d = (uint32_t)(((hi | e[limb]) >> (lo & 31)) & ((1u << (top - lo + 1)) - 1));
    const int tz = keyexp_ctz(d);                              // bit `top` is set: d != 0
    digit = d >> tz;
    return lo + tz;
}

// Number of windows of an exponent of `bits` bits and the low bit of the first (-1 and 0 windows for a zero exponent).
// The kernels' work counters use it; the schedule is the one the exponentiation loops walk.
KEYEXP_HD int keyexp_count(const uint32_t* e, int bits, int& first_lo) {
    int n = 0, top = keyexp_top(e, bits - 1);
    first_lo = -1;
    while (top >= 0) {
        uint32_t d;
        const int lo = keyexp_window(e, top, d);
        if (n++ == 0) first_lo = lo;
        top = keyexp_top(e, lo - 1);
    }
    return n;
}

// Slot order of a class whose exponent is a key-row value: units stable-sorted by `rows[u]`, each row's run padded to a
// multiple of `pad` slots (the groups per warp of every kernel the order serves, powers of two) with ORDER_PAD | (the run's
// first unit), so that every slot of a warp names a unit of the same row.  Writes the order and returns its length, at
// most units + (rows in use) * (pad - 1).  `count` is scratch of `nrows` entries.
inline size_t keyexp_order(const uint32_t* rows, size_t units, uint32_t nrows, size_t pad, uint32_t* count, uint32_t* order) {
    for (uint32_t r = 0; r < nrows; r++) count[r] = 0;
    for (size_t u = 0; u < units; u++) count[rows[u]]++;
    size_t len = 0;
    for (uint32_t r = 0; r < nrows; r++) {                     // count[r] becomes the first slot of row r's run
        const size_t n = count[r];
        count[r] = (uint32_t)len;
        len += (n + pad - 1) / pad * pad;
    }
    for (size_t u = 0; u < units; u++) order[count[rows[u]]++] = (uint32_t)u;
    // count[r] is now one past the last unit of row r's run; the run starts at the previous row's padded end
    size_t s = 0;
    for (uint32_t r = 0; r < nrows; r++) {
        if (count[r] == s) continue;                           // row not in use
        const uint32_t first = order[s];
        for (s = count[r]; s % pad; s++) order[s] = ORDER_PAD | first;
    }
    return len;
}

}  // namespace tecdsa
