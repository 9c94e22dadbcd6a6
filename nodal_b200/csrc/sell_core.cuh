// Per-entry rules of the SELL-32 entry encodings (sparse.cuh), written once for the CUDA kernels
// (spmv.cu) and for the host harness the CPU tests compile with g++ (tests/host_check/sell_host.cpp).
//
// wide:    int32 column + double value per stored entry (12 B).
// compact: int16 (column - row) + uint8 index into a table of at most 256 distinct value bit
//          patterns, sorted by bit pattern (3 B).  Lossless: decode(encode(v)) has v's bits.
// Padding inside a row stores the row itself with value +0.0; the tail lanes of the last slice
// (rows >= n) store column n - 1, which is a valid column whose offset fits int16 (>= -31).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SELLC_HD __host__ __device__ __forceinline__
#else
#include <string.h>
#define SELLC_HD static inline
#endif

constexpr int SELL_DICT_MAX = 256;   // entries of the compact value table (uint8 index)

// The bit pattern a value is compared and sorted by: +0.0 and -0.0, and NaNs with different
// payloads, are different values.
SELLC_HD uint64_t sell_bits(double v) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t u;
    memcpy(&u, &v, sizeof(u));
    return u;
#endif
}

SELLC_HD double sell_from_bits(uint64_t u) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double v;
    memcpy(&v, &u, sizeof(v));
    return v;
#endif
}

// Column stored for entry slot k of row r (r may be a tail lane, r >= n): the CSR column when the
// row has that entry, otherwise the padding column.
SELLC_HD int32_t sell_pad_col(int64_t r, int32_t n) { return r < n ? (int32_t)r : n - 1; }

SELLC_HD bool sell_offset_fits(int32_t c, int64_t r) {
    const int64_t d = (int64_t)c - r;
    return d >= -32768 && d <= 32767;
}

SELLC_HD int16_t sell_encode_col(int32_t c, int64_t r) { return (int16_t)((int64_t)c - r); }
SELLC_HD int32_t sell_decode_col(int16_t d, int64_t r) { return (int32_t)(r + d); }

// Index of bit pattern u in the sorted table dict[0..nd) (u must be in it).
SELLC_HD uint8_t sell_encode_val(const uint64_t* dict, int nd, uint64_t u) {
    int lo = 0, hi = nd - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (dict[mid] < u) lo = mid + 1;
        else hi = mid;
    }
    return (uint8_t)lo;
}
