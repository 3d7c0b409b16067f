// Reductions the plotting side of recoup runs over a finished profile matrix (SURVEY 8f, N4):
//   calcPlotProfiles   apply(x$profile, 2, mean|median) with sd|mad bands, optional log2(x + 1)
//                      (/root/reference/R/plot.R:949-990)
//   orderProfiles      apply(x$profile, 1, sum|max|mean) and sort(..., index.return=TRUE)
//                      (plot.R:1035-1150)
//   heat-map scale     quantile(x$profile, 0.95 ...) (plot.R:513-545), type 7
// The matrix is column-major  n_rows x n_cols  with leading dimension ld, as rcp_profile_matrix
// leaves it on the device.  Means and sums are plain streaming reductions (one CTA per column,
// one thread per row); medians, orderings and quantiles go through CUB's radix sort on
// order-preserving 64-bit keys.
#include <cub/device/device_radix_sort.cuh>

#include <cmath>
#include <utility>

#include "rcp_internal.cuh"

namespace rcp {
namespace {

constexpr int TPB = 256;
constexpr unsigned long long KEY_NAN = ~0ull;

__device__ __forceinline__ double scaled(double x, bool log2_scale) {
    return log2_scale ? log2(x + 1.0) : x;
}

// double -> u64 whose unsigned order is the numeric order; -0 == +0; NaN after everything
__device__ __forceinline__ unsigned long long ordered_key(double x) {
    if (x != x) return KEY_NAN;
    const unsigned long long b = (unsigned long long)__double_as_longlong(x + 0.0);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
    if (k == KEY_NAN) return nan("");
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// R accumulates sums and means in long double (summary.c); a plain double sum of a few hundred
// bin means differs from that in the last bits, which is enough to reorder near-tied rows.  The
// sums here are carried as unevaluated pairs hi + lo (error-free TwoSum), so that the value
// handed back is the correctly rounded exact sum in all but pathological cases -- the same
// double R's 64-bit-mantissa accumulator rounds to.
struct DD {
    double hi, lo;
};
__device__ __forceinline__ DD dd_add(DD a, double x) {
    const double s = a.hi + x;
    const double bb = s - a.hi;
    const double err = (a.hi - (s - bb)) + (x - bb);
    return {s, a.lo + err};
}
__device__ __forceinline__ DD dd_merge(DD a, DD b) {
    DD r = dd_add(a, b.hi);
    r.lo += b.lo;
    return r;
}
__device__ __forceinline__ double dd_value(DD a) { return a.hi + a.lo; }
// (hi + lo) / n, correctly rounded in practice
__device__ __forceinline__ double dd_div(DD a, double n) {
    const double s = a.hi + a.lo;
    const double rest = (a.hi - s) + a.lo;
    const double q = s / n;
    const double r = fma(-q, n, s) + rest;
    return q + r / n;
}

__device__ __forceinline__ DD block_sum(DD v, DD* sh) {
    for (int d = 16; d > 0; d >>= 1) {
        DD o;
        o.hi = __shfl_xor_sync(0xffffffffu, v.hi, d);
        o.lo = __shfl_xor_sync(0xffffffffu, v.lo, d);
        v = dd_merge(v, o);
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    DD t = sh[0];
    for (int k = 1; k < TPB / 32; k++) t = dd_merge(t, sh[k]);      // same order in every thread
    return t;
}

// One CTA per column: mean and sd (n - 1), both from exact-sum accumulators.
__global__ void __launch_bounds__(TPB)
col_mean_sd_kernel(const double* __restrict__ m, int64_t n_rows, int64_t ld, int log2_scale,
                   double* __restrict__ center, double* __restrict__ spread) {
    __shared__ DD sh[TPB / 32];
    const double* col = m + (int64_t)blockIdx.x * ld;
    const bool lg = log2_scale != 0;
    DD s = {0.0, 0.0};
    for (int64_t i = threadIdx.x; i < n_rows; i += TPB) s = dd_add(s, scaled(col[i], lg));
    const double mean = dd_div(block_sum(s, sh), (double)n_rows);
    DD q = {0.0, 0.0};
    for (int64_t i = threadIdx.x; i < n_rows; i += TPB) {
        const double d = scaled(col[i], lg) - mean;
        q = dd_add(q, d * d);
    }
    const double ss = dd_value(block_sum(q, sh));
    if (threadIdx.x == 0) {
        center[blockIdx.x] = mean;
        spread[blockIdx.x] = n_rows > 1 ? sqrt(ss / (double)(n_rows - 1)) : nan("");
    }
}

// what: 0 sum, 1 max, 2 mean -- one thread per row, columns walked in order
__global__ void __launch_bounds__(TPB)
row_stat_kernel(const double* __restrict__ m, int64_t n_rows, int64_t n_cols, int64_t ld, int what,
                double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n_rows) return;
    const double* p = m + i;
    if (what == 1) {
        double best = p[0];
        bool bad = best != best;
        for (int64_t c = 1; c < n_cols; c++) {
            const double v = p[c * ld];
            bad |= v != v;
            best = v > best ? v : best;
        }
        out[i] = bad ? nan("") : best;
        return;
    }
    DD s = {0.0, 0.0};
    for (int64_t c = 0; c < n_cols; c++) s = dd_add(s, p[c * ld]);
    out[i] = what == 2 ? dd_div(s, (double)n_cols) : dd_value(s);
}

// keys of a vector for sort(v, decreasing)$ix: ascending radix order of these keys, ties stable
__global__ void __launch_bounds__(TPB)
order_keys_kernel(const double* __restrict__ v, int64_t n, int decreasing,
                  unsigned long long* __restrict__ keys, int32_t* __restrict__ idx,
                  unsigned long long* __restrict__ n_nan) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    unsigned long long k = ordered_key(v[i]);
    if (k == KEY_NAN) atomicAdd(n_nan, 1ull);
    else if (decreasing) k = ~k;          // a number's key is never 0, so ~k is never KEY_NAN
    keys[i] = k;
    idx[i] = (int32_t)(i + 1);
}

// every cell of the matrix as a key (optionally |x - center[col]|), with its column id
__global__ void __launch_bounds__(TPB)
cell_keys_kernel(const double* __restrict__ m, int64_t n_rows, int64_t n_cols, int64_t ld,
                 int log2_scale, const double* __restrict__ center /* nullable */,
                 unsigned long long* __restrict__ keys, uint32_t* __restrict__ col_id /* nullable */,
                 unsigned long long* __restrict__ n_nan) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n_rows * n_cols) return;
    const int64_t c = i / n_rows, r = i - c * n_rows;
    double x = scaled(m[c * ld + r], log2_scale != 0);
    if (center) x = fabs(x - center[c]);
    const unsigned long long k = ordered_key(x);
    if (k == KEY_NAN) atomicAdd(n_nan, 1ull);
    keys[i] = k;
    if (col_id) col_id[i] = (uint32_t)c;
}

// widths of reads as keys; also used to count the reads not wider than a limit
__global__ void __launch_bounds__(TPB)
width_keys_kernel(int64_t n, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                  unsigned long long* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i < n) keys[i] = ordered_key((double)end[i] - (double)start[i] + 1.0);
}
__global__ void __launch_bounds__(TPB)
count_le_kernel(int64_t n, const unsigned long long* __restrict__ keys, const double* __restrict__ limit,
                unsigned long long* __restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    const bool le = i < n && !(key_value(keys[i]) > *limit);
    const unsigned m = __ballot_sync(0xffffffffu, le);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (unsigned long long)__popc(m));
}

// median of every sorted column segment (R: mean of the two middle values for even n)
__global__ void __launch_bounds__(TPB)
col_median_kernel(const unsigned long long* __restrict__ sorted, int64_t n_rows, int64_t n_cols,
                  double factor, double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (c >= n_cols) return;
    const unsigned long long* s = sorted + c * n_rows;
    const double lo = key_value(s[(n_rows - 1) / 2]), hi = key_value(s[n_rows / 2]);
    const double last = key_value(s[n_rows - 1]);           // NaN sorts last: NA propagates
    out[c] = (last != last) ? nan("") : factor * ((n_rows & 1) ? lo : (lo + hi) / 2.0);
}

// quantile type 7 on sorted keys: index = 1 + (n - 1) p; (1 - h) x[lo] + h x[hi]
__global__ void quantile_kernel(const unsigned long long* __restrict__ sorted, int64_t n,
                                const double* __restrict__ probs, int k, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const double index = (double)(n - 1) * probs[j];
    const double lo = floor(index), hi = ceil(index);
    const double xl = key_value(sorted[(int64_t)lo]), xh = key_value(sorted[(int64_t)hi]);
    const double h = index - lo;
    out[j] = (index > lo && xh != xl) ? (1.0 - h) * xl + h * xh : xl;
}

int sort_keys_u64(unsigned long long*& keys, int64_t n) {
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 values in one sort");
    unsigned long long* alt = nullptr;
    RCP_TRY(dalloc(&alt, (size_t)n));
    cub::DoubleBuffer<unsigned long long> buf(keys, alt);
    size_t tmp_bytes = 0;
    RCP_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, buf, (int)n, 0, 64, g_ctx.stream));
    uint8_t* tmp = nullptr;
    RCP_TRY(dalloc(&tmp, tmp_bytes));
    RCP_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, buf, (int)n, 0, 64, g_ctx.stream));
    g_ctx.launches += 9;
    dfree(tmp);
    if (buf.Current() != keys) std::swap(keys, alt);
    dfree(alt);
    return RCP_OK;
}

template <class V>
int sort_pairs(unsigned long long*& keys, V*& vals, int64_t n, int begin_bit, int end_bit) {
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 values in one sort");
    unsigned long long* kalt = nullptr;
    V* valt = nullptr;
    RCP_TRY(dalloc(&kalt, (size_t)n));
    RCP_TRY(dalloc(&valt, (size_t)n));
    cub::DoubleBuffer<unsigned long long> kb(keys, kalt);
    cub::DoubleBuffer<V> vb(vals, valt);
    size_t tmp_bytes = 0;
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, kb, vb, (int)n, begin_bit, end_bit,
                                             g_ctx.stream));
    uint8_t* tmp = nullptr;
    RCP_TRY(dalloc(&tmp, tmp_bytes));
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, kb, vb, (int)n, begin_bit, end_bit,
                                             g_ctx.stream));
    g_ctx.launches += 1 + (end_bit - begin_bit + 7) / 8;
    dfree(tmp);
    if (kb.Current() != keys) std::swap(keys, kalt);
    if (vb.Current() != vals) std::swap(vals, valt);
    dfree(kalt);
    dfree(valt);
    return RCP_OK;
}

// the same pairs, keyed the other way round: stable sort of the column ids carrying the keys
int sort_by_column(uint32_t*& col_id, unsigned long long*& keys, int64_t n, int col_bits) {
    uint32_t* calt = nullptr;
    unsigned long long* kalt = nullptr;
    RCP_TRY(dalloc(&calt, (size_t)n));
    RCP_TRY(dalloc(&kalt, (size_t)n));
    cub::DoubleBuffer<uint32_t> cb(col_id, calt);
    cub::DoubleBuffer<unsigned long long> kb(keys, kalt);
    size_t tmp_bytes = 0;
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, cb, kb, (int)n, 0, col_bits,
                                             g_ctx.stream));
    uint8_t* tmp = nullptr;
    RCP_TRY(dalloc(&tmp, tmp_bytes));
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, cb, kb, (int)n, 0, col_bits,
                                             g_ctx.stream));
    g_ctx.launches += 1 + (col_bits + 7) / 8;
    dfree(tmp);
    if (cb.Current() != col_id) std::swap(col_id, calt);
    if (kb.Current() != keys) std::swap(keys, kalt);
    dfree(calt);
    dfree(kalt);
    return RCP_OK;
}

struct MatIn {
    DevIn<double> in;
    int init(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int mem) {
        if (n_rows < 0 || n_cols < 0 || ld < n_rows || (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE))
            return fail(RCP_ERR_ARG, "matrix: bad shape, leading dimension or mem kind");
        if (n_rows > 0 && n_cols > 0 && m == nullptr) return fail(RCP_ERR_ARG, "matrix: NULL pointer");
        const size_t span = n_cols > 0 ? (size_t)(n_cols - 1) * (size_t)ld + (size_t)n_rows : 0;
        return in.init(m, span, mem);
    }
};

// result vector: computed on the device, delivered where the caller wants it
struct VecOut {
    double* dev = nullptr;
    double* user = nullptr;
    size_t n = 0;
    int mem = RCP_MEM_DEVICE;
    int init(double* out, size_t count, int mem_kind) {
        user = out;
        n = count;
        mem = mem_kind;
        if (mem == RCP_MEM_DEVICE) {
            dev = out;
            return RCP_OK;
        }
        return dalloc(&dev, count);
    }
    int finish() {
        if (mem == RCP_MEM_HOST && n > 0) {
            RCP_CUDA(cudaMemcpyAsync(user, dev, n * sizeof(double), cudaMemcpyDeviceToHost, g_ctx.stream));
            RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        }
        return RCP_OK;
    }
    ~VecOut() {
        if (mem == RCP_MEM_HOST) dfree(dev);
    }
};

int column_medians(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int log2_scale,
                   const double* center, double factor, double* out) {
    const int64_t n = n_rows * n_cols;
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "median profile: more than 2^31-1 cells");
    unsigned long long* keys = nullptr;
    uint32_t* col = nullptr;
    unsigned long long* n_nan = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)n));
    RCP_TRY(dalloc(&col, (size_t)n));
    RCP_TRY(dalloc(&n_nan, 1));
    RCP_CUDA(cudaMemsetAsync(n_nan, 0, 8, g_ctx.stream));
    cell_keys_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(
        m, n_rows, n_cols, ld, log2_scale, center, keys, col, n_nan);
    RCP_LAUNCHED();
    int rc = sort_pairs(keys, col, n, 0, 64);           // by value ...
    int col_bits = 1;
    while ((1ll << col_bits) < n_cols) col_bits++;
    if (rc == RCP_OK) rc = sort_by_column(col, keys, n, col_bits);      // ... then (stable) by column
    if (rc == RCP_OK) {
        col_median_kernel<<<(unsigned)((n_cols + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(
            keys, n_rows, n_cols, factor, out);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess) rc = fail(RCP_ERR_CUDA, "col_median_kernel launch failed");
    }
    dfree(keys);
    dfree(col);
    dfree(n_nan);
    return rc;
}

}  // namespace

int sort_pairs_u64_i32(unsigned long long*& keys, int32_t*& vals, int64_t n) {
    return sort_pairs(keys, vals, n, 0, 64);
}

}  // namespace rcp

using namespace rcp;

extern "C" {

int rcp_matrix_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int stat,
                           int log2_scale, int mem, double* center, double* spread) {
    RCP_TRY(require_ready());
    if (stat != RCP_STAT_MEAN && stat != RCP_STAT_MEDIAN) return fail(RCP_ERR_ARG, "col_profile: bad stat");
    if (center == nullptr || spread == nullptr) return fail(RCP_ERR_ARG, "col_profile: NULL output");
    MatIn in;
    RCP_TRY(in.init(m, n_rows, n_cols, ld, mem));
    if (n_cols == 0) return RCP_OK;
    if (n_rows == 0) return fail(RCP_ERR_ARG, "col_profile: the matrix has no rows");
    VecOut c, s;
    RCP_TRY(c.init(center, (size_t)n_cols, mem));
    RCP_TRY(s.init(spread, (size_t)n_cols, mem));
    if (stat == RCP_STAT_MEAN) {
        col_mean_sd_kernel<<<(unsigned)n_cols, TPB, 0, g_ctx.stream>>>(in.in.ptr, n_rows, ld, log2_scale,
                                                                       c.dev, s.dev);
        RCP_LAUNCHED();
    } else {
        RCP_TRY(column_medians(in.in.ptr, n_rows, n_cols, ld, log2_scale, nullptr, 1.0, c.dev));
        // mad(x) = 1.4826 * median(|x - median(x)|)
        RCP_TRY(column_medians(in.in.ptr, n_rows, n_cols, ld, log2_scale, c.dev, 1.4826, s.dev));
    }
    RCP_TRY(c.finish());
    RCP_TRY(s.finish());
    return RCP_OK;
}

int rcp_matrix_row_stat(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int what, int mem,
                        double* out) {
    RCP_TRY(require_ready());
    if (what < RCP_ROW_SUM || what > RCP_ROW_MEAN) return fail(RCP_ERR_ARG, "row_stat: bad statistic");
    if (out == nullptr) return fail(RCP_ERR_ARG, "row_stat: NULL output");
    MatIn in;
    RCP_TRY(in.init(m, n_rows, n_cols, ld, mem));
    if (n_rows == 0) return RCP_OK;
    if (n_cols == 0) return fail(RCP_ERR_ARG, "row_stat: the matrix has no columns");
    VecOut o;
    RCP_TRY(o.init(out, (size_t)n_rows, mem));
    row_stat_kernel<<<(unsigned)((n_rows + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(in.in.ptr, n_rows, n_cols,
                                                                                   ld, what, o.dev);
    RCP_LAUNCHED();
    return o.finish();
}

int rcp_order(const double* v, int64_t n, int decreasing, int mem, int32_t* ix, int64_t* n_out) {
    RCP_TRY(require_ready());
    if (n < 0 || (n > 0 && (v == nullptr || ix == nullptr)) || (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE))
        return fail(RCP_ERR_ARG, "order: bad argument");
    if (n_out) *n_out = 0;
    if (n == 0) return RCP_OK;
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "order: more than 2^31-1 values");
    DevIn<double> in;
    RCP_TRY(in.init(v, (size_t)n, mem));
    unsigned long long* keys = nullptr;
    int32_t* idx = nullptr;
    unsigned long long* n_nan = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)n));
    RCP_TRY(dalloc(&idx, (size_t)n));
    RCP_TRY(dalloc(&n_nan, 1));
    RCP_CUDA(cudaMemsetAsync(n_nan, 0, 8, g_ctx.stream));
    order_keys_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(in.ptr, n, decreasing, keys,
                                                                                 idx, n_nan);
    RCP_LAUNCHED();
    int rc = sort_pairs(keys, idx, n, 0, 64);
    unsigned long long h_nan = 0;
    if (rc == RCP_OK) {
        cudaError_t e = cudaMemcpyAsync(ix, idx, (size_t)n * 4,
                                        mem == RCP_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                        g_ctx.stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(&h_nan, n_nan, 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "order: copy back failed: %s", cudaGetErrorString(e));
    }
    dfree(keys);
    dfree(idx);
    dfree(n_nan);
    if (rc == RCP_OK && n_out) *n_out = n - (int64_t)h_nan;
    return rc;
}

int rcp_reads_width_quantile(int64_t n, const int32_t* start, const int32_t* end, double prob, int mem,
                             double* quantile_out, int64_t* n_le_out) {
    RCP_TRY(require_ready());
    if (n <= 0 || start == nullptr || end == nullptr || quantile_out == nullptr ||
        (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE))
        return fail(RCP_ERR_ARG, "width_quantile: bad argument");
    if (!(prob >= 0.0 && prob <= 1.0)) return fail(RCP_ERR_ARG, "width_quantile: 'probs' outside [0,1]");
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "width_quantile: more than 2^31-1 reads");
    DevIn<int32_t> d_start, d_end;
    RCP_TRY(d_start.init(start, (size_t)n, mem));
    RCP_TRY(d_end.init(end, (size_t)n, mem));
    unsigned long long* keys = nullptr;
    unsigned long long* count = nullptr;
    double *d_prob = nullptr, *d_out = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)n));
    RCP_TRY(dalloc(&count, 1));
    RCP_TRY(dalloc(&d_prob, 1));
    RCP_TRY(dalloc(&d_out, 1));
    RCP_CUDA(cudaMemsetAsync(count, 0, 8, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_prob, &prob, 8, cudaMemcpyHostToDevice, g_ctx.stream));
    const unsigned blocks = (unsigned)((n + TPB - 1) / TPB);
    width_keys_kernel<<<blocks, TPB, 0, g_ctx.stream>>>(n, d_start.ptr, d_end.ptr, keys);
    RCP_LAUNCHED();
    int rc = sort_keys_u64(keys, n);
    unsigned long long h_count = 0;
    if (rc == RCP_OK) {
        quantile_kernel<<<1, 64, 0, g_ctx.stream>>>(keys, n, d_prob, 1, d_out);
        count_le_kernel<<<blocks, TPB, 0, g_ctx.stream>>>(n, keys, d_out, count);
        g_ctx.launches += 2;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(quantile_out, d_out, 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_count, count, 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "width_quantile failed: %s", cudaGetErrorString(e));
    }
    dfree(keys);
    dfree(count);
    dfree(d_prob);
    dfree(d_out);
    if (rc == RCP_OK && n_le_out) *n_le_out = (int64_t)h_count;
    return rc;
}

int rcp_matrix_quantile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, const double* probs,
                        int k, int mem, double* out /* host, k */) {
    RCP_TRY(require_ready());
    if (k < 0 || (k > 0 && (probs == nullptr || out == nullptr))) return fail(RCP_ERR_ARG, "quantile: bad argument");
    for (int j = 0; j < k; j++)
        if (!(probs[j] >= 0.0 && probs[j] <= 1.0)) return fail(RCP_ERR_ARG, "quantile: 'probs' outside [0,1]");
    MatIn in;
    RCP_TRY(in.init(m, n_rows, n_cols, ld, mem));
    const int64_t n = n_rows * n_cols;
    if (k == 0) return RCP_OK;
    if (n == 0) return fail(RCP_ERR_ARG, "quantile: empty matrix");
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "quantile: more than 2^31-1 cells");
    unsigned long long* keys = nullptr;
    unsigned long long* n_nan = nullptr;
    double *d_probs = nullptr, *d_out = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)n));
    RCP_TRY(dalloc(&n_nan, 1));
    RCP_TRY(dalloc(&d_probs, (size_t)k));
    RCP_TRY(dalloc(&d_out, (size_t)k));
    RCP_CUDA(cudaMemsetAsync(n_nan, 0, 8, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_probs, probs, (size_t)k * 8, cudaMemcpyHostToDevice, g_ctx.stream));
    cell_keys_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(in.in.ptr, n_rows, n_cols, ld, 0,
                                                                                nullptr, keys, nullptr, n_nan);
    RCP_LAUNCHED();
    int rc = sort_keys_u64(keys, n);
    unsigned long long h_nan = 0;
    if (rc == RCP_OK) {
        quantile_kernel<<<(k + 63) / 64, 64, 0, g_ctx.stream>>>(keys, n, d_probs, k, d_out);
        g_ctx.launches++;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, (size_t)k * 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_nan, n_nan, 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "quantile failed: %s", cudaGetErrorString(e));
    }
    dfree(keys);
    dfree(n_nan);
    dfree(d_probs);
    dfree(d_out);
    if (rc == RCP_OK && h_nan > 0)
        return fail(RCP_ERR_DATA, "quantile: missing values and NaN's not allowed if 'na.rm' is FALSE");
    return rc;
}

}  // extern "C"
