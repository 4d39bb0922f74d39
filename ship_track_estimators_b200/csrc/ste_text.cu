// ste_text.cu - the CLI's text files for whole fleets on the device (np.savetxt's "%.18e", main_cli.py:146-167).
//
// Two launches around an inclusive scan the caller runs (torch.cumsum):
//   text_convert_kernel  one thread per value: gathers it from its table, converts it exactly (ste_text.cuh) and
//                        stores its 19 digits, a meta word and its length with separator;
//   text_write_kernel    one thread per value: formats it into shared memory at its offset within the block's
//                        contiguous span of the output, then the block copies that span out in order.
#include <cstdio>

#include "ste_text.cuh"
#include "../../include/ste_ukf.h"

namespace ste {
int report_error(int code, const char *what);   // ste_ukf.cu: sets ste_last_error()
int report_launch(const char *what);

constexpr int kTextThreads = 256;
static_assert(text::kMaxValueBytes == STE_TEXT_MAX_VALUE_BYTES, "header and kernel disagree on the longest field");

struct TextTables {
    SteTextTable t[STE_TEXT_MAX_TABLES];
    int32_t n_tables;
    int64_t n_segments;   // n_items * n_tables
};

__global__ void __launch_bounds__(kTextThreads) text_convert_kernel(const TextTables tb, const int64_t *__restrict__ value_start,
                                                                    int64_t n_values, uint64_t *__restrict__ digits,
                                                                    int32_t *__restrict__ meta, int32_t *__restrict__ length) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_values) return;
    int64_t lo = 0, hi = tb.n_segments;   // the last segment g with value_start[g] <= v
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(value_start + mid) <= v) lo = mid;
        else hi = mid;
    }
    const int item = (int)(lo / tb.n_tables);
    const SteTextTable &t = tb.t[lo % tb.n_tables];
    const int64_t local = v - __ldg(value_start + lo);
    const int64_t row = local / t.n_cols;
    const int col = (int)(local - row * t.n_cols);
    const int64_t plane = (row / t.row_div) * t.row_stride + t.plane[col];
    const double x = __ldg(t.base + plane * t.ld + __ldg(t.track + item));
    uint64_t d;
    int32_t m;
    text::convert(x, d, m);
    if (col == t.n_cols - 1) m |= text::kMetaNewline;
    digits[v] = d;
    meta[v] = m;
    length[v] = text::field_length(m) + 1;
}

__global__ void __launch_bounds__(kTextThreads) text_write_kernel(int64_t n_values, const uint64_t *__restrict__ digits,
                                                                  const int32_t *__restrict__ meta, const int64_t *__restrict__ end,
                                                                  uint8_t *__restrict__ out) {
    __shared__ char buf[kTextThreads * text::kMaxValueBytes];
    const int64_t v0 = (int64_t)blockIdx.x * kTextThreads;
    const int64_t v_last = min(v0 + kTextThreads, n_values) - 1;
    const int64_t base = end[v0] - (text::field_length(meta[v0]) + 1);
    const int64_t v = v0 + threadIdx.x;
    if (v <= v_last) {
        const int32_t m = meta[v];
        const int64_t start = end[v] - (text::field_length(m) + 1);
        text::format_field(digits[v], m, buf + (start - base));
    }
    __syncthreads();
    const int64_t span = end[v_last] - base;
    for (int64_t i = threadIdx.x; i < span; i += kTextThreads) out[base + i] = (uint8_t)buf[i];
}

}  // namespace ste

using namespace ste;

extern "C" {

int ste_text_convert_f64(const SteTextTable *tables, int32_t n_tables, int32_t n_items, const int64_t *value_start, int64_t n_values,
                         uint64_t *digits, int32_t *meta, int32_t *length, void *stream) {
    if (n_tables < 1 || n_tables > STE_TEXT_MAX_TABLES) return report_error(STE_ERR_INVALID_ARG, "n_tables outside [1, STE_TEXT_MAX_TABLES]");
    if (n_items < 0 || n_values < 0) return report_error(STE_ERR_INVALID_ARG, "negative item or value count");
    if (!tables || !value_start || !digits || !meta || !length) return report_error(STE_ERR_INVALID_ARG, "missing array");
    TextTables tb{};
    for (int k = 0; k < n_tables; ++k) {
        const SteTextTable &t = tables[k];
        if (!t.base || !t.track) return report_error(STE_ERR_INVALID_ARG, "table without source or track array");
        if (t.n_tracks < 0) return report_error(STE_ERR_INVALID_ARG, "negative track count in a table");
        if (t.ld < t.n_tracks) return report_error(STE_ERR_INVALID_ARG, "ld < n_tracks");
        if (t.n_cols < 1 || t.n_cols > STE_TEXT_MAX_COLS) return report_error(STE_ERR_INVALID_ARG, "n_cols outside [1, STE_TEXT_MAX_COLS]");
        if (t.row_stride < 1 || t.row_div < 1) return report_error(STE_ERR_INVALID_ARG, "row_stride and row_div must be >= 1");
        for (int c = 0; c < t.n_cols; ++c)
            if (t.plane[c] < 0 || t.plane[c] >= t.row_stride) return report_error(STE_ERR_INVALID_ARG, "plane index outside [0, row_stride)");
        tb.t[k] = t;
    }
    if (n_values == 0) return STE_OK;
    if (n_items == 0) return report_error(STE_ERR_INVALID_ARG, "values without items");
    const int64_t blocks = (n_values + kTextThreads - 1) / kTextThreads;
    if (blocks > 0x7fffffffll) return report_error(STE_ERR_UNSUPPORTED, "more than 2^31 blocks of values: split the tables");
    tb.n_tables = n_tables;
    tb.n_segments = (int64_t)n_items * n_tables;
    text_convert_kernel<<<(unsigned)blocks, kTextThreads, 0, (cudaStream_t)stream>>>(tb, value_start, n_values, digits, meta, length);
    return report_launch("text_convert_kernel");
}

int ste_text_write(int64_t n_values, const uint64_t *digits, const int32_t *meta, const int64_t *end, uint8_t *out, int64_t out_bytes,
                   void *stream) {
    if (n_values < 0) return report_error(STE_ERR_INVALID_ARG, "negative value count");
    if (!digits || !meta || !end || !out) return report_error(STE_ERR_INVALID_ARG, "missing array");
    if (out_bytes < 0 || out_bytes / STE_TEXT_MAX_VALUE_BYTES < n_values)
        return report_error(STE_ERR_INVALID_ARG, "output buffer smaller than STE_TEXT_MAX_VALUE_BYTES per value");
    if (n_values == 0) return STE_OK;
    const int64_t blocks = (n_values + kTextThreads - 1) / kTextThreads;
    if (blocks > 0x7fffffffll) return report_error(STE_ERR_UNSUPPORTED, "more than 2^31 blocks of values: split the tables");
    text_write_kernel<<<(unsigned)blocks, kTextThreads, 0, (cudaStream_t)stream>>>(n_values, digits, meta, end, out);
    return report_launch("text_write_kernel");
}

}  // extern "C"
