// TEST-ONLY: compiles the per-entry rules of the SELL entry encodings (nodal_b200/csrc/sell_core.cuh)
// for the CPU and builds a SELL-32 matrix from CSR the way sell_from_csr does, in both encodings,
// so `pytest -m "not gpu"` can check the choice (offsets that fit int16, at most 256 distinct value
// bit patterns with the +0.0 of the padding) and that decoding the compact entries gives the wide
// ones bit for bit.  The distinct values are counted with std::set here, with hash sets on the device.
// Not part of the product library.
#include <stdint.h>

#include <set>

#include "../../nodal_b200/csrc/sell_core.cuh"

// Census: returns 1 when the matrix goes compact; then dict[0..*ndict) is the sorted table.
// *fits: every offset col - row fits int16.
extern "C" int sellh_plan(int32_t n, const int32_t* indptr, const int32_t* indices, const double* data,
                          int32_t* fits, uint64_t* dict, int32_t* ndict) {
    std::set<uint64_t> seen{sell_bits(0.0)};
    *fits = 1;
    for (int32_t r = 0; r < n; ++r)
        for (int32_t j = indptr[r]; j < indptr[r + 1]; ++j) {
            if (!sell_offset_fits(indices[j], r)) *fits = 0;
            seen.insert(sell_bits(data[j]));
        }
    *ndict = (int32_t)seen.size();
    if (n == 0 || !*fits || seen.size() > (size_t)SELL_DICT_MAX) return 0;
    int k = 0;
    for (uint64_t u : seen) dict[k++] = u;
    return 1;
}

// Fills the slices (slice_w: exclusive scan of the widths, [nslices + 1]) in both encodings.
extern "C" void sellh_fill(int32_t n, const int32_t* indptr, const int32_t* indices, const double* data,
                           const uint32_t* slice_w, const uint64_t* dict, int32_t ndict, int32_t* cols, double* vals,
                           int16_t* dcol, uint8_t* vidx) {
    const int32_t nslices = (n + 31) / 32;
    for (int32_t s = 0; s < nslices; ++s)
        for (int lane = 0; lane < 32; ++lane) {
            const int64_t r = (int64_t)s * 32 + lane;
            const int32_t b = r < n ? indptr[r] : 0, e = r < n ? indptr[r + 1] : 0;
            for (uint32_t k = 0; k < slice_w[s + 1] - slice_w[s]; ++k) {
                int32_t c = sell_pad_col(r, n);
                double v = 0.0;
                if (b + (int32_t)k < e) { c = indices[b + k]; v = data[b + k]; }
                const int64_t i = ((int64_t)slice_w[s] + k) * 32 + lane;
                cols[i] = c;
                vals[i] = v;
                if (dict) {
                    dcol[i] = sell_encode_col(c, r);
                    vidx[i] = sell_encode_val(dict, ndict, sell_bits(v));
                }
            }
        }
}

// The (column, value) a reader sees for every compact entry.
extern "C" void sellh_decode(int32_t n, const uint32_t* slice_w, const int16_t* dcol, const uint8_t* vidx,
                             const uint64_t* dict, int32_t* cols, double* vals) {
    const int32_t nslices = (n + 31) / 32;
    for (int32_t s = 0; s < nslices; ++s)
        for (int lane = 0; lane < 32; ++lane) {
            const int64_t r = (int64_t)s * 32 + lane;
            for (uint32_t k = 0; k < slice_w[s + 1] - slice_w[s]; ++k) {
                const int64_t i = ((int64_t)slice_w[s] + k) * 32 + lane;
                cols[i] = sell_decode_col(dcol[i], r);
                vals[i] = sell_from_bits(dict[vidx[i]]);
            }
        }
}
