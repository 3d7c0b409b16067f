// Reductions the plotting side of recoup runs over a finished profile matrix (SURVEY 8f, N4):
//   calcPlotProfiles   apply(x$profile, 2, mean|median) with sd|mad bands, optional log2(x + 1)
//                      (/root/reference/R/plot.R:949-990)
//   calcDesignPlotProfiles  the same per design level (rows grouped by an integer code)
//   orderProfiles      apply(x$profile, 1, sum|max|mean) and sort(..., index.return=TRUE)
//                      (plot.R:1035-1150)
//   heat-map scale     quantile(x$profile, 0.95 ...) (plot.R:513-545), type 7
// The matrix is column-major  n_rows x n_cols  with leading dimension ld, as rcp_profile_matrix
// leaves it on the device.  The curve and band of calcPlotProfiles are computed per group of rows
// (calcDesignPlotProfiles: one curve per design level; a single group is calcPlotProfiles): means
// are chunked exact-sum reductions, medians a segmented radix sort.  Row sums are plain streaming
// reductions (one thread per row); orderings and quantiles go through the library's radix sort
// (sort.cu) on order-preserving 64-bit keys.
#include <cub/device/device_segmented_radix_sort.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include <algorithm>
#include <climits>
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
// Once the plain sum hi is not finite (an infinite or NaN cell, or an overflow) the pair is
// {hi, 0}: TwoSum's error term would be inf - inf = NaN and turn a +-Inf sum into NaN.
struct DD {
    double hi, lo;
};
__device__ __forceinline__ DD dd_add(DD a, double x) {
    const double s = a.hi + x;
    const double bb = s - a.hi;
    const double err = (a.hi - (s - bb)) + (x - bb);
    return {s, isfinite(s) ? a.lo + err : 0.0};
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
    const double q = s / n;
    if (!isfinite(s)) return q;
    const double rest = (a.hi - s) + a.lo;
    const double r = fma(-q, n, s) + rest;
    return q + r / n;
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

// every cell of the matrix as a key
__global__ void __launch_bounds__(TPB)
cell_keys_kernel(const double* __restrict__ m, int64_t n_rows, int64_t n_cols, int64_t ld,
                 unsigned long long* __restrict__ keys, unsigned long long* __restrict__ n_nan) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n_rows * n_cols) return;
    const int64_t c = i / n_rows, r = i - c * n_rows;
    const unsigned long long k = ordered_key(m[c * ld + r]);
    if (k == KEY_NAN) atomicAdd(n_nan, 1ull);
    keys[i] = k;
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

// quantile type 7 on sorted keys, R's quantile.default operation for operation:
//   index <- 1 + (n - 1) * p; lo <- floor(index); hi <- ceiling(index) (1-based);
//   h <- index - lo; (1 - h) * x[lo] + h * x[hi] where index > lo and x[hi] != x[lo].
// Every product and sum is rounded on its own (no FMA contraction), as R rounds them.
__global__ void quantile_kernel(const unsigned long long* __restrict__ sorted, int64_t n,
                                const double* __restrict__ probs, int k, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const double index = __dadd_rn(1.0, __dmul_rn((double)(n - 1), probs[j]));
    const double lo = floor(index), hi = ceil(index);
    const double xl = key_value(sorted[(int64_t)lo - 1]), xh = key_value(sorted[(int64_t)hi - 1]);
    const double h = index - lo;
    out[j] = (index > lo && xh != xl) ? __dadd_rn(__dmul_rn(1.0 - h, xl), __dmul_rn(h, xh)) : xl;
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

// ------------------------------------------------------------------ per-group column profile --
// Row i belongs to group codes[i] (1..G; <= 0 excluded).  A stable radix sort of the codes gives
// the rows grouped by code, ascending within each group; start[g] (g = 1..G+1) is the first sorted
// position whose code is >= g, so group g - 1 (0-based) holds grouped rows
// [start[g] - start[1], start[g + 1] - start[1]) and start[1] rows are excluded.  Unless G == 1 and
// no row is excluded, the matrix is copied once into that row order (n_inc x n_cols, column-major),
// which makes every (column, group) segment contiguous.
//
// Mean and sd: a warp sums a chunk of GP_CHUNK grouped rows of one column, whatever groups it
// spans, and leaves one exact (DD) partial per (group, chunk) piece.  Pieces are stored at slot
// g + k (group g, chunk k): consecutive pieces increase g or k or both, so the slots are distinct,
// and a group's pieces are the slots g + first_chunk(g) .. g + last_chunk(g).  A second kernel
// merges each (column, group)'s pieces in chunk order.  One 10^6-row group and 10^6 one-row groups
// are the same amount of work per warp, and the launches are the same for every G.
// Median and mad: order-preserving keys of every cell, one segmented radix sort per statistic
// with (column, group) segments, and the middle values.
constexpr int GP_CHUNK = 2048;
constexpr int GP_WARPS = TPB / 32;
constexpr unsigned GP_MAX_GRID_Y = 65535;

__host__ __device__ __forceinline__ int64_t group_off(const int64_t* start, int g) { return start[g + 1] - start[1]; }
// 0-based group of grouped row r (gkey: the sorted codes from the first grouped row on, or NULL)
__device__ __forceinline__ int group_of(const uint32_t* gkey, int64_t r) { return gkey ? (int)gkey[r] - 1 : 0; }

__global__ void __launch_bounds__(TPB)
group_sort_keys_kernel(const int32_t* __restrict__ codes, int64_t n, uint32_t* __restrict__ key,
                       int32_t* __restrict__ row) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const int32_t c = codes[i];
    key[i] = c > 0 ? (uint32_t)c : 0u;
    row[i] = (int32_t)i;
}

// start[1..G+1] from the sorted codes (skey NULL: every row in group 1); *bad = 1 on a code > G
__global__ void __launch_bounds__(TPB)
group_bounds_kernel(const uint32_t* __restrict__ skey, int64_t n, int G, int64_t* __restrict__ start,
                    unsigned* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i > n) return;
    const int64_t top = (int64_t)G + 1;
    auto key = [&](int64_t j) -> int64_t { return skey ? (skey[j] < (uint32_t)top ? (int64_t)skey[j] : top) : 1; };
    const int64_t prev = i == 0 ? 0 : key(i - 1);
    const int64_t cur = i == n ? top : key(i);
    if (i < n && skey && skey[i] > (uint32_t)G) *bad = 1u;
    for (int64_t g = prev + 1; g <= cur; g++) start[g] = i;
}

// place[i]: grouped row of source row i, or -1 when the row is excluded
__global__ void __launch_bounds__(TPB)
group_place_kernel(const int32_t* __restrict__ srow, int64_t n, const int64_t* __restrict__ start,
                   int64_t* __restrict__ place) {
    const int64_t p = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (p >= n) return;
    const int64_t n_excl = start[1];
    place[srow[p]] = p >= n_excl ? p - n_excl : -1;
}

// the copy: source rows read in order (coalesced), each written to its grouped row
__global__ void __launch_bounds__(TPB)
group_scatter_kernel(const double* __restrict__ m, int64_t n_rows, int64_t n_cols, int64_t ld,
                     const int64_t* __restrict__ place, int64_t n_inc, double* __restrict__ x) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t to = place[i];
    if (to < 0) return;
    for (int64_t c = blockIdx.y; c < n_cols; c += gridDim.y) x[c * n_inc + to] = m[c * ld + i];
}

__device__ __forceinline__ DD shfl_dd(DD v, int src) {
    return {__shfl_sync(0xffffffffu, v.hi, src), __shfl_sync(0xffffffffu, v.lo, src)};
}
// sum over the warp in a fixed order, the value of lane 0 broadcast
__device__ __forceinline__ DD warp_dd_sum(DD v) {
    for (int d = 16; d > 0; d >>= 1) {
        DD o;
        o.hi = __shfl_xor_sync(0xffffffffu, v.hi, d);
        o.lo = __shfl_xor_sync(0xffffffffu, v.lo, d);
        v = dd_merge(v, o);
    }
    return shfl_dd(v, 0);
}

// PASS 0: pieces of sum(x); PASS 1: pieces of sum((x - center)^2).  One warp per (chunk, column).
template <int PASS>
__global__ void __launch_bounds__(TPB)
group_chunk_sum_kernel(const double* __restrict__ x, int64_t L, int64_t n_inc, int64_t n_chunks, int64_t n_cols,
                       int G, const uint32_t* __restrict__ gkey, const int64_t* __restrict__ start,
                       int log2_scale, const double* __restrict__ center, int64_t P, DD* __restrict__ part) {
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * GP_WARPS + (threadIdx.x >> 5);
    if (k >= n_chunks) return;
    const bool lg = log2_scale != 0;
    const int64_t a = k * GP_CHUNK, b = min(a + GP_CHUNK, n_inc);
    const int first = group_of(gkey, a);
    for (int64_t c = blockIdx.y; c < n_cols; c += gridDim.y) {
        const double* col = x + c * L;
        DD* pc = part + c * P;
        auto emit = [&](int g, DD v) { pc[g + k] = v; };
        int cur = first;
        DD acc = {0.0, 0.0};
        for (int64_t base = a; base < b; base += 32) {
            const int64_t r = base + lane;
            const int last = (int)min((int64_t)31, b - 1 - base);
            const bool valid = lane <= last;
            const int g = valid ? group_of(gkey, r) : INT_MAX;
            double v = 0.0;
            if (valid) {
                v = scaled(col[r], lg);
                if (PASS == 1) {
                    const double d = v - center[c * G + g];
                    v = d * d;
                }
            }
            const int g_last = __shfl_sync(0xffffffffu, g, last);
            if (g_last == cur) {            // the codes are sorted: the whole step is group cur
                acc = dd_add(acc, v);
                continue;
            }
            const DD tot = warp_dd_sum(acc);
            DD s = {v, 0.0};                // inclusive scan within each run of equal groups
            for (int d = 1; d < 32; d <<= 1) {
                const DD o = {__shfl_up_sync(0xffffffffu, s.hi, d), __shfl_up_sync(0xffffffffu, s.lo, d)};
                const int go = __shfl_up_sync(0xffffffffu, g, d);
                if (lane >= d && go == g) s = dd_merge(o, s);
            }
            if (g == cur) s = dd_merge(tot, s);
            else if (lane == 0) emit(cur, tot);       // group cur ended with the previous step
            const int g_next = __shfl_down_sync(0xffffffffu, g, 1);
            if (valid && lane < last && g_next != g) emit(g, s);
            acc = lane == last ? s : DD{0.0, 0.0};
            cur = g_last;
        }
        const DD tot = warp_dd_sum(acc);
        if (lane == 0) emit(cur, tot);
    }
}

// PASS 0: center = mean; PASS 1: spread = sd (n - 1).  One thread per (group, column).
template <int PASS>
__global__ void __launch_bounds__(TPB)
group_merge_kernel(int64_t n_cols, int G, const int64_t* __restrict__ start, int64_t P, const DD* __restrict__ part,
                   double* __restrict__ out) {
    const int64_t s = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (s >= n_cols * G) return;
    const int64_t c = s / G;
    const int g = (int)(s - c * G);
    const int64_t lo = group_off(start, g), n = group_off(start, g + 1) - lo;
    DD t = {0.0, 0.0};
    if (n > 0) {
        const DD* pc = part + c * P + g;
        for (int64_t k = lo / GP_CHUNK; k <= (lo + n - 1) / GP_CHUNK; k++) t = dd_merge(t, pc[k]);
    }
    if (PASS == 0) out[s] = n > 0 ? dd_div(t, (double)n) : nan("");
    else out[s] = n > 1 ? sqrt(dd_value(t) / (double)(n - 1)) : nan("");
}

// keys of the grouped cells (|x - center| when center is given), n_inc x n_cols compact
__global__ void __launch_bounds__(TPB)
group_cell_keys_kernel(const double* __restrict__ x, int64_t L, int64_t n_inc, int64_t n_cols, int G,
                       const uint32_t* __restrict__ gkey, int log2_scale, const double* __restrict__ center,
                       unsigned long long* __restrict__ keys) {
    const int64_t r = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (r >= n_inc) return;
    const int g = group_of(gkey, r);
    for (int64_t c = blockIdx.y; c < n_cols; c += gridDim.y) {
        double v = scaled(x[c * L + r], log2_scale != 0);
        if (center) v = fabs(v - center[c * G + g]);
        keys[c * n_inc + r] = ordered_key(v);
    }
}

// median of every sorted (group, column) segment, times factor (R: mean of the two middle values)
__global__ void __launch_bounds__(TPB)
group_median_kernel(const unsigned long long* __restrict__ sorted, int64_t n_inc, int64_t n_cols, int G,
                    const int64_t* __restrict__ start, double factor, double* __restrict__ out) {
    const int64_t s = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (s >= n_cols * G) return;
    const int64_t c = s / G;
    const int g = (int)(s - c * G);
    const int64_t lo = group_off(start, g), n = group_off(start, g + 1) - lo;
    if (n == 0) {
        out[s] = nan("");
        return;
    }
    const unsigned long long* q = sorted + c * n_inc + lo;
    const double a = key_value(q[(n - 1) / 2]), b = key_value(q[n / 2]);
    const double last = key_value(q[n - 1]);           // NaN sorts last: NA propagates
    out[s] = (last != last) ? nan("") : factor * ((n & 1) ? a : (a + b) / 2.0);
}

// segment s = (column s / G, group s % G) of the compact key array
struct SegBegin {
    const int64_t* start;
    int64_t n_inc;
    int G;
    __host__ __device__ int operator()(int s) const {
        const int c = s / G, g = s - c * G;
        return (int)(c * n_inc + group_off(start, g));
    }
};
struct SegEnd {
    const int64_t* start;
    int64_t n_inc;
    int G;
    __host__ __device__ int operator()(int s) const {
        const int c = s / G, g = s - c * G;
        return (int)(c * n_inc + group_off(start, g + 1));
    }
};

int group_medians(const double* x, int64_t L, int64_t n_inc, int64_t n_cols, int G, const uint32_t* gkey,
                  const int64_t* start, int log2_scale, const double* center, double factor, double* out) {
    const int64_t n = n_inc * n_cols;
    const int n_seg = (int)(n_cols * G);
    unsigned long long *keys = nullptr, *alt = nullptr;
    uint8_t* tmp = nullptr;
    int rc = RCP_OK;
    if (n > 0) {
        RCP_TRY(dalloc(&keys, (size_t)n));
        rc = dalloc(&alt, (size_t)n);
        if (rc == RCP_OK) {
            const dim3 grid((unsigned)((n_inc + TPB - 1) / TPB), (unsigned)std::min<int64_t>(n_cols, GP_MAX_GRID_Y));
            group_cell_keys_kernel<<<grid, TPB, 0, g_ctx.stream>>>(x, L, n_inc, n_cols, G, gkey, log2_scale, center,
                                                                   keys);
            g_ctx.launches++;
            cub::DoubleBuffer<unsigned long long> buf(keys, alt);
            auto begin = thrust::make_transform_iterator(thrust::make_counting_iterator(0), SegBegin{start, n_inc, G});
            auto end = thrust::make_transform_iterator(thrust::make_counting_iterator(0), SegEnd{start, n_inc, G});
            size_t tmp_bytes = 0;
            cudaError_t e = cudaGetLastError();
            if (e == cudaSuccess)
                e = cub::DeviceSegmentedRadixSort::SortKeys(nullptr, tmp_bytes, buf, (int)n, n_seg, begin, end, 0, 64,
                                                            g_ctx.stream);
            if (e == cudaSuccess) rc = dalloc(&tmp, tmp_bytes);
            if (e == cudaSuccess && rc == RCP_OK) {
                e = cub::DeviceSegmentedRadixSort::SortKeys(tmp, tmp_bytes, buf, (int)n, n_seg, begin, end, 0, 64,
                                                            g_ctx.stream);
                g_ctx.launches += 11;       // one pass per radix digit of the 64-bit keys
            }
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "group median: %s", cudaGetErrorString(e));
            if (buf.Current() != keys) std::swap(keys, alt);
        }
    }
    if (rc == RCP_OK) {
        group_median_kernel<<<(unsigned)((n_seg + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(keys, n_inc, n_cols, G,
                                                                                          start, factor, out);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess) rc = fail(RCP_ERR_CUDA, "group_median_kernel launch failed");
    }
    dfree(tmp);
    dfree(alt);
    dfree(keys);
    return rc;
}

int group_mean_sd(const double* x, int64_t L, int64_t n_inc, int64_t n_cols, int G, const uint32_t* gkey,
                  const int64_t* start, int log2_scale, double* center, double* spread) {
    const int64_t n_chunks = (n_inc + GP_CHUNK - 1) / GP_CHUNK;
    const int64_t P = (int64_t)G + n_chunks;          // slots g + k
    DD* part = nullptr;
    RCP_TRY(dalloc(&part, (size_t)(P * n_cols)));
    const dim3 grid((unsigned)((n_chunks + GP_WARPS - 1) / GP_WARPS), (unsigned)std::min<int64_t>(n_cols, GP_MAX_GRID_Y));
    const unsigned merge_blocks = (unsigned)((n_cols * G + TPB - 1) / TPB);
    int rc = RCP_OK;
    if (n_chunks > 0) {
        group_chunk_sum_kernel<0><<<grid, TPB, 0, g_ctx.stream>>>(x, L, n_inc, n_chunks, n_cols, G, gkey, start,
                                                                  log2_scale, nullptr, P, part);
        g_ctx.launches++;
    }
    group_merge_kernel<0><<<merge_blocks, TPB, 0, g_ctx.stream>>>(n_cols, G, start, P, part, center);
    g_ctx.launches++;
    if (n_chunks > 0) {
        group_chunk_sum_kernel<1><<<grid, TPB, 0, g_ctx.stream>>>(x, L, n_inc, n_chunks, n_cols, G, gkey, start,
                                                                  log2_scale, center, P, part);
        g_ctx.launches++;
    }
    group_merge_kernel<1><<<merge_blocks, TPB, 0, g_ctx.stream>>>(n_cols, G, start, P, part, spread);
    g_ctx.launches++;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "group mean/sd launch failed: %s", cudaGetErrorString(e));
    dfree(part);
    return rc;
}

// shapes are checked by the caller; codes NULL: one group of every row
int group_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, const int32_t* codes, int G,
                      int stat, int log2_scale, int mem, double* center, double* spread) {
    MatIn in;
    RCP_TRY(in.init(m, n_rows, n_cols, ld, mem));
    DevIn<int32_t> d_codes;
    RCP_TRY(d_codes.init(codes, (size_t)n_rows, mem));
    VecOut c, s;
    RCP_TRY(c.init(center, (size_t)(G * n_cols), mem));
    RCP_TRY(s.init(spread, (size_t)(G * n_cols), mem));
    uint32_t* skey = nullptr;
    int32_t* srow = nullptr;
    int64_t* start = nullptr;
    unsigned* bad = nullptr;
    int64_t* place = nullptr;
    double* grouped = nullptr;
    int rc = dalloc(&start, (size_t)G + 2);
    if (rc == RCP_OK) rc = dalloc(&bad, 1);
    if (rc == RCP_OK && codes) {
        rc = dalloc(&skey, (size_t)n_rows);
        if (rc == RCP_OK) rc = dalloc(&srow, (size_t)n_rows);
        if (rc == RCP_OK) {
            group_sort_keys_kernel<<<(unsigned)((n_rows + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(d_codes.ptr, n_rows,
                                                                                                    skey, srow);
            g_ctx.launches++;
            rc = sort_pairs(skey, srow, n_rows, 0, 32);     // stable: ascending rows within a group
        }
    }
    int64_t n_excl = 0;
    if (rc == RCP_OK) {
        cudaError_t e = cudaMemsetAsync(bad, 0, sizeof(unsigned), g_ctx.stream);
        if (e == cudaSuccess) {
            group_bounds_kernel<<<(unsigned)((n_rows + TPB) / TPB), TPB, 0, g_ctx.stream>>>(skey, n_rows, G, start, bad);
            g_ctx.launches++;
            e = cudaGetLastError();
        }
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "group bounds: %s", cudaGetErrorString(e));
    }
    if (rc == RCP_OK && codes) {
        unsigned h_bad = 0;
        const FetchItem items[2] = {{start + 1, &n_excl, 8}, {bad, &h_bad, 4}};
        rc = fetch_and_sync(items, 2);
        if (rc == RCP_OK && h_bad) rc = fail(RCP_ERR_DATA, "group_col_profile: a code is greater than n_groups");
    }
    const int64_t n_inc = n_rows - n_excl;
    const double* x = in.in.ptr;
    int64_t L = ld;
    if (rc == RCP_OK && codes && (G > 1 || n_excl > 0)) {
        rc = dalloc(&place, (size_t)n_rows);
        if (rc == RCP_OK) rc = dalloc(&grouped, (size_t)std::max<int64_t>(n_inc * n_cols, 1));
        if (rc == RCP_OK) {
            const unsigned blocks = (unsigned)((n_rows + TPB - 1) / TPB);
            group_place_kernel<<<blocks, TPB, 0, g_ctx.stream>>>(srow, n_rows, start, place);
            group_scatter_kernel<<<dim3(blocks, (unsigned)std::min<int64_t>(n_cols, GP_MAX_GRID_Y)), TPB, 0,
                                   g_ctx.stream>>>(x, n_rows, n_cols, ld, place, n_inc, grouped);
            g_ctx.launches += 2;
            const cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "group copy: %s", cudaGetErrorString(e));
        }
        x = grouped;
        L = n_inc;
    }
    const uint32_t* gkey = skey ? skey + n_excl : nullptr;
    if (rc == RCP_OK) {
        if (stat == RCP_STAT_MEAN) {
            rc = group_mean_sd(x, L, n_inc, n_cols, G, gkey, start, log2_scale, c.dev, s.dev);
        } else {
            rc = group_medians(x, L, n_inc, n_cols, G, gkey, start, log2_scale, nullptr, 1.0, c.dev);
            // mad(x) = 1.4826 * median(|x - median(x)|)
            if (rc == RCP_OK) rc = group_medians(x, L, n_inc, n_cols, G, gkey, start, log2_scale, c.dev, 1.4826, s.dev);
        }
    }
    if (rc == RCP_OK) rc = c.finish();
    if (rc == RCP_OK) rc = s.finish();
    dfree(grouped);
    dfree(place);
    dfree(bad);
    dfree(start);
    dfree(srow);
    dfree(skey);
    return rc;
}

// the checks both entry points share, before any allocation
int col_profile_args(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int stat, int mem,
                     const double* center, const double* spread) {
    if (stat != RCP_STAT_MEAN && stat != RCP_STAT_MEDIAN) return fail(RCP_ERR_ARG, "col_profile: bad stat");
    if (center == nullptr || spread == nullptr) return fail(RCP_ERR_ARG, "col_profile: NULL output");
    if (n_rows < 0 || n_cols < 0 || ld < n_rows || (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE))
        return fail(RCP_ERR_ARG, "matrix: bad shape, leading dimension or mem kind");
    if (n_rows > 0 && n_cols > 0 && m == nullptr) return fail(RCP_ERR_ARG, "matrix: NULL pointer");
    return RCP_OK;
}
}  // namespace

}  // namespace rcp

using namespace rcp;

extern "C" {

int rcp_matrix_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int stat,
                           int log2_scale, int mem, double* center, double* spread) {
    RCP_TRY(require_ready());
    RCP_TRY(col_profile_args(m, n_rows, n_cols, ld, stat, mem, center, spread));
    if (n_cols == 0) return RCP_OK;
    if (n_rows == 0) return fail(RCP_ERR_ARG, "col_profile: the matrix has no rows");
    if (stat == RCP_STAT_MEDIAN && n_rows > 0x7fffffff / n_cols)
        return fail(RCP_ERR_UNSUPPORTED, "median profile: more than 2^31-1 cells");
    return group_col_profile(m, n_rows, n_cols, ld, nullptr, 1, stat, log2_scale, mem, center, spread);
}

int rcp_matrix_group_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, const int32_t* codes,
                                 int n_groups, int stat, int log2_scale, int mem, double* center, double* spread) {
    RCP_TRY(require_ready());
    RCP_TRY(col_profile_args(m, n_rows, n_cols, ld, stat, mem, center, spread));
    if (n_groups < 1) return fail(RCP_ERR_ARG, "col_profile: n_groups must be at least 1");
    if (n_rows == 0) return fail(RCP_ERR_ARG, "col_profile: the matrix has no rows");
    if (n_cols > 0 && n_rows > 0x7fffffff / n_cols)
        return fail(RCP_ERR_UNSUPPORTED, "col_profile: more than 2^31-1 cells");
    if ((int64_t)n_groups * n_cols > 0x7fffffff)
        return fail(RCP_ERR_UNSUPPORTED, "col_profile: n_groups x n_cols above 2^31-1");
    if (n_cols == 0) return RCP_OK;
    return group_col_profile(m, n_rows, n_cols, ld, codes, n_groups, stat, log2_scale, mem, center, spread);
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
    int rc = sort_keys(keys, n, 0, 64);
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
    cell_keys_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(in.in.ptr, n_rows, n_cols, ld,
                                                                                keys, n_nan);
    RCP_LAUNCHED();
    int rc = sort_keys(keys, n, 0, 64);
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
