// Profile-matrix kernels (sm_100a): binCoverageMatrix / baseCoverageMatrix / splitVector of the
// reference (/root/reference/R/profile.R:100-212, R/util.R:15-85).
//
//   bin_mean_kernel      persistent CTAs: bin edges from R's seed-42 rank table (util.R:74-80),
//                        segment staged by cp.async (double-buffered) and prefix-summed in
//                        place, bin sum = two shared-memory loads, fp64 mean, column-major
//   bin_median_kernel    1 CTA / region: exact median by value bisection
//   interp_kernel        regions shorter than the bin count (util.R:17-73): fmm spline or
//                        neighbourhood fill, one warp per flagged region
//   base_matrix_kernel   per-base matrix: counts -> fp64 tiled transpose (profile.R:100-151)
//
// Every kernel that reads coverage values is a template on the value type V of the handle:
// int32_t (reads: 64-bit integer sums) or float (signal tracks: fp64 sums; the words hold float
// bits).  The helpers below are the only places the two differ; for int32_t they are the casts
// the kernels always used.
//
// Each such kernel also has a storage type S: int32_t (4-byte words) or, for int32 counts of the
// split path that no tile could push past 65 535, uint16_t (cov_narrow).  The kernel reads the
// coverage's decision word once at entry and runs the matching instance of its body: the branch is
// uniform over the grid, and the host never waits for the word.

#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "r_rng.cuh"
#include "rcp_internal.cuh"

namespace rcp {

namespace {

constexpr int CTA = 256;
constexpr int WARPS = CTA / 32;

template <class V>
struct Val;
template <>
struct Val<int32_t> {
    using Sum = long long;
    using Key = int;                                    // median bisection over the values
    static constexpr int KEY_MIN = -0x7fffffff - 1, KEY_MAX = 0x7fffffff;
};
template <>
struct Val<float> {
    using Sum = double;
    using Key = unsigned;                               // order-preserving key of the float
    static constexpr unsigned KEY_MIN = 0u, KEY_MAX = 0xffffffffu;
};
// a staged word -> its term in a sum
template <class V>
__device__ __forceinline__ typename Val<V>::Sum word_sum(uint32_t w) {
    if constexpr (std::is_same<V, float>::value) return (double)__uint_as_float(w);
    else return (long long)w;
}
// a loaded word -> its value (int stays int)
template <class V>
__device__ __forceinline__ auto word_val(int w) {
    if constexpr (std::is_same<V, float>::value) return (double)__int_as_float(w);
    else return w;
}
template <class V>
__device__ __forceinline__ double word_double(int w) {
    if constexpr (std::is_same<V, float>::value) return (double)__int_as_float(w);
    else return (double)w;
}
// median keys: the value itself for int32; for float the bits with the sign flipped (positive)
// or all bits flipped (negative), so that unsigned order is float order (-0.0 never occurs)
template <class V>
__device__ __forceinline__ typename Val<V>::Key word_key(int w) {
    if constexpr (std::is_same<V, float>::value) {
        const unsigned u = (unsigned)w;
        return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    } else {
        return w;
    }
}
template <class V>
__device__ __forceinline__ double key_double(typename Val<V>::Key k) {
    if constexpr (std::is_same<V, float>::value)
        return (double)__uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
    else return (double)k;
}

// storage: log2 of the elements in 16 bytes, and the unsigned word a staged element is read as
template <class S>
constexpr int LOG_PER16 = sizeof(S) == 2 ? 3 : 2;
template <class S>
using Word = typename std::conditional<sizeof(S) == 2, uint16_t, uint32_t>::type;
// a staged 16-byte unit -> its term in a sum (8 counts of at most 65 535 fit 32 bits)
template <class V, class S>
__device__ __forceinline__ typename Val<V>::Sum unit_sum(uint4 x) {
    if constexpr (sizeof(S) == 2) {
        return (long long)(((x.x & 0xffffu) + (x.x >> 16)) + ((x.y & 0xffffu) + (x.y >> 16)) +
                           ((x.z & 0xffffu) + (x.z >> 16)) + ((x.w & 0xffffu) + (x.w >> 16)));
    } else {
        return (word_sum<V>(x.x) + word_sum<V>(x.y)) + (word_sum<V>(x.z) + word_sum<V>(x.w));
    }
}
// elements [q, q + 4) (q a multiple of 4) as loaded: 16 bytes, or 8 when narrow; widen4 unpacks them.
// The streaming loops keep rows packed in registers and, when narrow, put twice the rows in flight,
// so that a warp has as many bytes outstanding in either layout.
template <class S>
using Raw4 = typename std::conditional<sizeof(S) == 2, uint2, int4>::type;
__device__ __forceinline__ int4 widen4(int4 v) { return v; }
__device__ __forceinline__ int4 widen4(uint2 u) {
    return make_int4((int)(u.x & 0xffffu), (int)(u.x >> 16), (int)(u.y & 0xffffu), (int)(u.y >> 16));
}
template <class S>
__device__ __forceinline__ Raw4<S> load4_cs(const S* p) {
    return __ldcs(reinterpret_cast<const Raw4<S>*>(p));
}
template <class S>
__device__ __forceinline__ int4 load4_g(const S* p) {
    return widen4(__ldg(reinterpret_cast<const Raw4<S>*>(p)));
}
template <class S>
constexpr int ROWS_IN_FLIGHT = sizeof(S) == 2 ? 8 : 4;

// the part of a lane's four elements at or after a bin edge (c of them lie before it): for
// integers the row total minus the part before; for floats the sum of those elements, since
// tot - before loses the small ones beside a large one (1e20 + 7 - 1e20 == 0)
template <class V, class S, class A>
__device__ __forceinline__ S after_edge(S tot, S before, int c, A a0, A a1, A a2, A a3) {
    if constexpr (std::is_same<V, float>::value)
        return (S)(c <= 0 ? a0 : 0) + (c <= 1 ? a1 : 0) + (c <= 2 ? a2 : 0) + (c <= 3 ? a3 : 0);
    else return tot - before;
}

struct Seg {
    int a, b;   // [a, b) inside the region's coverage vector
};

__device__ __forceinline__ Seg segment_of(int L, int where, int f1, int f2) {
    Seg s;
    switch (where) {
        case RCP_WHERE_CENTER: s.a = f1; s.b = L - f2; break;          // profile.R:170
        case RCP_WHERE_UPSTREAM: s.a = 0; s.b = f1; break;              // profile.R:178
        case RCP_WHERE_DOWNSTREAM: s.a = L - f2; s.b = L; break;        // profile.R:185
        default: s.a = 0; s.b = L; break;                               // profile.R:159-162
    }
    if (s.a < 0) s.a = 0;
    if (s.b > L) s.b = L;
    if (s.b < s.a) s.b = s.a;
    return s;
}

struct BinArgs {
    const int32_t* cov;
    const unsigned long long* bound;   // Coverage::d_bound
    const int64_t* off;
    const int32_t* len;
    const uint8_t* is_null;
    const int* rank;          // device rank table of n bins
    int where, f1, f2, n;
    double scale;
    double* out;
    int64_t ld;
    int32_t* short_list;      // regions with segment shorter than n (for interp_kernel)
    unsigned int* short_count;
};

constexpr int STAGE_INTS = 12288;      // ints of one region staged in shared memory (48 KB)
constexpr int STAGE_MAX_BIN = 128;     // bins narrower than this use the staged path
constexpr int LONG_REGION_MIN = 16384; // wide-bin segments from this length on: bin_wide_kernel

// Sum of src[lo, hi) by one warp with 16-byte loads where the index is 4-aligned (src itself is
// 128-byte aligned: region offsets are multiples of 32 ints).
__device__ __forceinline__ long long warp_range_sum(const int32_t* __restrict__ src, int lo, int hi) {
    const int lane = threadIdx.x & 31;
    long long s = 0;
    const int a4 = (lo + 3) & ~3, b4 = hi & ~3;
    if (a4 >= b4) {
        for (int q = lo + lane; q < hi; q += 32) s += __ldg(src + q);
    } else {
        if (lo + lane < a4) s += __ldg(src + lo + lane);
        const int4* v = reinterpret_cast<const int4*>(src + a4);
        const int nv = (b4 - a4) >> 2;
        for (int q = lane; q < nv; q += 32) {
            const int4 x = __ldg(v + q);
            s += (long long)x.x + x.y + x.z + x.w;
        }
        if (b4 + lane < hi) s += __ldg(src + b4 + lane);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    return s;
}

// Median bins (sumStat = "median"): one CTA per region.  dynamic smem: edges[n + 1].
// (static shared memory lives in the kernel, so that the two instances of a body share it)
struct MedianSmem {
    int wcount[WARPS];
    int chunk_carry;
};
template <class V, class S>
__device__ __forceinline__ void bin_median_run(const BinArgs& p, MedianSmem& sm) {
    using K = typename Val<V>::Key;
    extern __shared__ __align__(16) int sh[];
    int* edges = sh;                    // n + 1
    auto& wcount = sm.wcount;
    auto& chunk_carry = sm.chunk_carry;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r = blockIdx.x;
    const int n = p.n;
    double* out = p.out + r;
    if (p.is_null[r]) {                 // profile.R:191-197: NULL -> zero row
        for (int i = tid; i < n; i += CTA) out[(int64_t)i * p.ld] = 0.0;
        return;
    }
    const int L = p.len[r];
    const Seg sg = segment_of(L, p.where, p.f1, p.f2);
    const int Ls = sg.b - sg.a;
    if (Ls < n) {                       // util.R:17: interpolation path, handled separately
        if (tid == 0) {
            if (Ls <= 0) {
                for (int i = 0; i < n; i++) out[(int64_t)i * p.ld] = 0.0;
            } else {
                p.short_list[atomicAdd(p.short_count, 1u)] = (int32_t)r;
            }
        }
        return;
    }
    // ---- bin edges: bin i has bsz + [rank[i] <= dif] elements (util.R:74-80) ----
    const int bsz = Ls / n, dif = Ls - bsz * n;
    if (dif == 0) {                     // equal bins: no rank table involved
        for (int i = tid; i <= n; i += CTA) edges[i] = sg.a + i * bsz;
        __syncthreads();
    } else {
        if (tid == 0) chunk_carry = 0;
        __syncthreads();
        for (int c0 = 0; c0 < n; c0 += CTA) {
            const int i = c0 + tid;
            const bool extra = (i < n) && (p.rank[i] <= dif);
            const unsigned bal = __ballot_sync(0xffffffffu, extra);
            if (lane == 0) wcount[warp] = __popc(bal);
            __syncthreads();
            int pre = chunk_carry;
            for (int w = 0; w < warp; w++) pre += wcount[w];
            pre += __popc(bal & ((1u << lane) - 1u));
            if (i < n) edges[i] = sg.a + i * bsz + pre;
            __syncthreads();
            if (tid == CTA - 1) chunk_carry = pre + (extra ? 1 : 0);
            __syncthreads();
        }
        if (tid == 0) edges[n] = sg.b;
        __syncthreads();
    }
    const S* src = reinterpret_cast<const S*>(p.cov) + p.off[r];
    // ---- median: groups of g lanes per bin, exact order statistics by value bisection ----
    int g = 1;
    while (g < 32 && g < bsz) g <<= 1;
    const int per_warp = 32 / g;
    const int sub = lane / g, li = lane % g;
    for (int b0 = warp * per_warp; b0 < n; b0 += WARPS * per_warp) {
        const int i = b0 + sub;
        const bool ok = i < n;
        const int lo = ok ? edges[i] : 0, hi = ok ? edges[i + 1] : 0;
        const int cnt = hi - lo;
        // k-th smallest = least v with #{x <= v} >= k+1
        K vmin = Val<V>::KEY_MAX, vmax = Val<V>::KEY_MIN;
        for (int q = lo + li; q < hi; q += g) {
            const K v = word_key<V>(__ldg(src + q));
            vmin = min(vmin, v);
            vmax = max(vmax, v);
        }
        for (int d = g >> 1; d > 0; d >>= 1) {
            vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, d));
            vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
        }
        const int k1 = (cnt - 1) / 2, k2 = cnt / 2;
        K res[2];
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const int k = t == 0 ? k1 : k2;
            K a = vmin, b = vmax;            // answer in [a, b]
            // every lane of the WARP iterates the same number of times (the shuffles are
            // warp-wide): bound by the warp-wide maximum range
            K span = ok ? (b - a) : 0;
            for (int d = 16; d > 0; d >>= 1) span = max(span, __shfl_xor_sync(0xffffffffu, span, d));
            while (span > 0) {
                const K mid = a + ((b - a) >> 1);
                int c = 0;
                for (int q = lo + li; q < hi; q += g) c += (word_key<V>(__ldg(src + q)) <= mid);
                for (int d = g >> 1; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
                if (a < b) {
                    if (c >= k + 1) b = mid;
                    else a = mid + 1;
                }
                span >>= 1;
            }
            res[t] = a;
        }
        if (ok && li == 0)
            out[(int64_t)i * p.ld] = p.scale * ((key_double<V>(res[0]) + key_double<V>(res[1])) * 0.5);
    }
}

template <class V>
__global__ void __launch_bounds__(CTA) bin_median_kernel(BinArgs p) {
    __shared__ MedianSmem sm;
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return bin_median_run<V, uint16_t>(p, sm);
    }
    bin_median_run<V, int32_t>(p, sm);
}

// ---- TMA (1-D bulk copy) + mbarrier helpers for the staging of bin_mean_kernel ----------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// global -> shared bulk copy by the TMA unit (one thread issues it; `bytes` a multiple of 16,
// both addresses 16-byte aligned); completion is signalled on `bar` as transaction bytes
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- mean bins: persistent, double-buffered ----------------------------------------------------
// One 32-byte descriptor per region (written by bin_desc_kernel), so that the main kernel does
// no divisions and loads nothing else per region:
//   x, y   offset of the region in the dense coverage (low / high word)
//   z, w   the segment [a, b) to bin (b <= a: NULL or empty -> zero row)
//   bsz, dif   bin width and the number of bins one base wider (util.R:74-80); bsz = 0: the
//              segment is shorter than the bin count (interpolation list)
//   lo_al, nvec   staging run (16-byte aligned first base, 16-byte units) when the whole segment is ONE
//              staged run of narrow bins -- only those are prefetched; nvec = 0 otherwise
struct __align__(16) BinDesc {
    int off_lo, off_hi, a, b;
    int bsz, dif, lo_al, nvec;
};

constexpr int BT = 256;                // threads of bin_mean_kernel
constexpr int BWARPS = BT / 32;

__global__ void __launch_bounds__(CTA)
bin_desc_kernel(int64_t R, const int64_t* __restrict__ off, const int32_t* __restrict__ len,
                const uint8_t* __restrict__ is_null, int where, int f1, int f2, int n,
                int buf_ints, BinDesc* __restrict__ desc, int32_t* __restrict__ long_list,
                unsigned int* __restrict__ long_count, const unsigned long long* __restrict__ bound) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= R) return;
    const bool narrow = cov_narrow(bound);
    const int sh = narrow ? 3 : 2;                      // log2 of the elements in a 16-byte unit
    const int cap = narrow ? (buf_ints >> 1) & ~3 : buf_ints;     // ints of one buffer of bin_mean_kernel
    Seg sg;
    sg.a = sg.b = 0;
    if (!is_null[r]) sg = segment_of(len[r], where, f1, f2);
    const uint64_t o = (uint64_t)off[r];
    BinDesc d;
    d.off_lo = (int)(uint32_t)o;
    d.off_hi = (int)(uint32_t)(o >> 32);
    d.a = sg.a;
    d.b = sg.b;
    const int Ls = sg.b - sg.a;
    d.bsz = Ls >= n ? Ls / n : 0;
    d.dif = Ls >= n ? Ls - d.bsz * n : 0;
    d.lo_al = sg.a & ~((1 << sh) - 1);
    d.nvec = 0;
    if (d.bsz > 0 && d.bsz < STAGE_MAX_BIN) {
        const int nvec = (sg.b - d.lo_al + (1 << sh) - 1) >> sh;
        if (nvec * 4 <= cap) d.nvec = nvec;             // 16 bytes per unit, 4 per int of the buffer
    }
    // a long region with wide bins (gene bodies run to megabases) would keep ONE CTA busy long
    // after the others have finished: its bins go to bin_wide_kernel, one warp per bin, spread
    // over the whole grid
    if (d.bsz >= STAGE_MAX_BIN && Ls >= LONG_REGION_MIN) {
        d.nvec = -1;
        long_list[atomicAdd(long_count, 1u)] = (int32_t)r;
    }
    desc[r] = d;
}

__device__ __forceinline__ BinDesc load_bin_desc(const BinDesc* __restrict__ p) {
    const int4 u = __ldg(reinterpret_cast<const int4*>(p));
    const int4 v = __ldg(reinterpret_cast<const int4*>(p) + 1);
    BinDesc d;
    d.off_lo = u.x; d.off_hi = u.y; d.a = u.z; d.b = u.w;
    d.bsz = v.x; d.dif = v.y; d.lo_al = v.z; d.nvec = v.w;
    return d;
}

// Persistent CTAs walk the regions.  Narrow bins (< 128 bases, the usual case: TSS windows,
// flanks): the segment is staged in shared memory and every bin is summed from there by a small
// group of threads with 16-byte shared-memory loads and 64-bit sums.  The staging
// copy of the NEXT region -- one TMA bulk copy (cp.async.bulk, up to 48 KB) issued by a single
// thread into the second buffer, completion on an mbarrier -- and the descriptor of the region
// after it are issued before the current region is processed, so HBM latency hides behind the
// arithmetic and no thread spends instructions on the copy.
// Wide bins: one warp per bin, 16-byte global loads.  Segments shorter than the bin count go
// to the interpolation list (util.R:17).
constexpr int NBUF_MAX = 8;

struct MeanSmem {
    int wcount[BWARPS];
    int chunk_carry;
    __align__(8) uint64_t full_bar[NBUF_MAX];     // one per staging buffer
    BinDesc ring[NBUF_MAX];                       // descriptor of the region in each buffer
};
template <class V, class ST>
__device__ __forceinline__ void bin_mean_run(const BinArgs& p, const BinDesc* __restrict__ desc, int64_t R,
                                             int buf_ints, int nbuf, MeanSmem& sm) {
    using S = typename Val<V>::Sum;
    constexpr int ESH = LOG_PER16<ST>, E = 1 << ESH;     // elements per 16-byte unit
    if (sizeof(ST) == 2) {      // a region takes half the bytes: twice the buffers in the same shared memory
        buf_ints = (buf_ints >> 1) & ~3;
        nbuf = min(2 * nbuf, NBUF_MAX);
    }
    extern __shared__ __align__(16) int sh[];
    int* edges = sh;                                         // n + 1 (unequal bins only)
    uint32_t* bufs = reinterpret_cast<uint32_t*>(sh + ((p.n + 1 + 3) & ~3));
    auto& wcount = sm.wcount;
    auto& chunk_carry = sm.chunk_carry;
    auto& full_bar = sm.full_bar;
    auto& ring = sm.ring;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = p.n;
    const int64_t step = gridDim.x;
    int64_t r = blockIdx.x;
    if (r >= R) return;
    if (tid == 0) {
        for (int k = 0; k < nbuf; k++) mbar_init(&full_bar[k], 1);
        fence_proxy_async();                // make the initialised barriers visible to the TMA unit
    }
    __syncthreads();
    BinDesc none;
    none.off_lo = none.off_hi = none.a = none.b = none.bsz = none.dif = none.lo_al = none.nvec = 0;

    auto src_of = [&](const BinDesc& d) {
        return reinterpret_cast<const ST*>(p.cov) + (int64_t)(((uint64_t)(uint32_t)d.off_hi << 32) | (uint32_t)d.off_lo);
    };
    // thread 0 starts the copy of one region into buffer `which` (regions that are not one staged
    // run just complete the barrier phase) and publishes its descriptor beside it
    auto issue = [&](const BinDesc& d, int which) {
        if (tid != 0) return;
        ring[which] = d;
        uint64_t* bar = &full_bar[which];
        if (d.nvec > 0) {
            const uint32_t bytes = (uint32_t)d.nvec * 16u;
            fence_proxy_async();            // earlier generic reads of this buffer are ordered first
            mbar_arrive_expect_tx(bar, bytes);
            tma_load_1d(bufs + (size_t)which * buf_ints, src_of(d) + d.lo_al, bytes, bar);
        } else {
            mbar_arrive(bar);
        }
    };

    // The staging buffers form a ring of nbuf: the copies of the next nbuf - 1 regions are in
    // flight while one region is processed (HBM latency is hidden by DEPTH: the per-region work
    // is light), and the descriptor of the region after those is already in registers.
    auto desc_at = [&](int64_t k) {         // descriptor of this CTA's k-th region
        const int64_t rr = blockIdx.x + k * step;
        return rr < R ? load_bin_desc(desc + rr) : none;
    };
    for (int k = 0; k < nbuf - 1; k++) issue(desc_at(k), k);
    BinDesc dq = desc_at(nbuf - 1);         // next to be issued
    uint32_t parity = 0;                    // bit k: phase of buffer k's barrier
    for (int64_t it = 0;; it++) {
        const int cur = (int)(it % nbuf);
        issue(dq, (int)((it + nbuf - 1) % nbuf));
        dq = desc_at(it + nbuf);
        uint32_t* stage = bufs + (size_t)cur * buf_ints;
        mbar_wait(&full_bar[cur], (parity >> cur) & 1u);    // this region's copy has landed
        parity ^= 1u << cur;
        const BinDesc d = ring[cur];
        double* out = p.out + r;
        const int Ls = d.b - d.a;
        if (Ls <= 0) {                      // NULL coverage -> zero row (profile.R:191-197)
            for (int i = tid; i < n; i += BT) out[(int64_t)i * p.ld] = 0.0;
        } else if (d.bsz == 0) {            // util.R:17: interpolation path, handled separately
            if (tid == 0) p.short_list[atomicAdd(p.short_count, 1u)] = (int32_t)r;
        } else if (d.nvec < 0) {            // long region, wide bins: bin_wide_kernel
        } else {
            // ---- bin edges: bin i has bsz + [rank[i] <= dif] elements (util.R:74-80) ----
            const int bsz = d.bsz, dif = d.dif;
            const bool equal = dif == 0;    // equal bins: edge i = a + i * bsz, no table
            if (!equal) {
                if (tid == 0) chunk_carry = 0;
                __syncthreads();
                for (int c0 = 0; c0 < n; c0 += BT) {
                    const int i = c0 + tid;
                    const bool extra = (i < n) && (p.rank[i] <= dif);
                    const unsigned bal = __ballot_sync(0xffffffffu, extra);
                    if (lane == 0) wcount[warp] = __popc(bal);
                    __syncthreads();
                    int pre = chunk_carry;
                    for (int w = 0; w < warp; w++) pre += wcount[w];
                    pre += __popc(bal & ((1u << lane) - 1u));
                    if (i < n) edges[i] = d.a + i * bsz + pre;
                    __syncthreads();
                    if (tid == BT - 1) chunk_carry = pre + (extra ? 1 : 0);
                    __syncthreads();
                }
                if (tid == 0) edges[n] = d.b;
                __syncthreads();
            }
            auto edge = [&](int i) { return equal ? d.a + i * bsz : edges[i]; };
            const ST* src = src_of(d);
            const Word<ST>* staged = reinterpret_cast<const Word<ST>*>(stage);
            if (bsz < STAGE_MAX_BIN) {
                const bool preloaded = d.nvec > 0;
                const int bins_per_chunk = preloaded ? n : max(1, ((buf_ints << (ESH - 2)) - E) / (bsz + 1));
                for (int bin0 = 0; bin0 < n; bin0 += bins_per_chunk) {
                    const int bin1 = min(n, bin0 + bins_per_chunk);
                    const int lo_al = preloaded ? d.lo_al : (edge(bin0) & ~(E - 1));
                    const int nvec = preloaded ? d.nvec : ((edge(bin1) - lo_al + E - 1) >> ESH);
                    if (!preloaded) {       // several runs per region: staged here, no overlap
                        __syncthreads();
                        const int4* gsrc = reinterpret_cast<const int4*>(src + lo_al);
                        for (int i = tid; i < nvec; i += BT)
                            reinterpret_cast<int4*>(stage)[i] = __ldg(gsrc + i);
                        __syncthreads();
                    }
                    // g threads per bin (a power of two that divides the warp): each walks its
                    // share of the bin in the staged data -- scalar up to the first 16-byte
                    // boundary, 16-byte loads after it, scalar tail -- with 64-bit sums; the g
                    // parts meet by shuffles.  About 1.5 instructions per base.
                    const int nb = bin1 - bin0;
                    int g = 1;
                    while (g < 32 && 2 * g * nb <= BT) g <<= 1;
                    const int part = tid & (g - 1);
                    for (int b0 = bin0; b0 < bin1; b0 += BT / g) {      // whole warps stay together
                        const int b = b0 + tid / g;
                        S s64 = 0;
                        int eb0 = 0, eb1 = 1;
                        if (b < bin1) {
                            eb0 = edge(b);
                            eb1 = edge(b + 1);
                            const int blen = eb1 - eb0;
                            const int share = (blen + g - 1) / g;
                            int q = eb0 - lo_al + part * share;
                            const int qe = min(q + share, eb1 - lo_al);
                            while (q < qe && (q & (E - 1))) s64 += word_sum<V>(staged[q++]);
                            for (; q + E <= qe; q += E) s64 += unit_sum<V, ST>(*reinterpret_cast<const uint4*>(staged + q));
                            while (q < qe) s64 += word_sum<V>(staged[q++]);
                        }
                        for (int dd = g >> 1; dd > 0; dd >>= 1) s64 += __shfl_xor_sync(0xffffffffu, s64, dd);
                        if (b < bin1 && part == 0)
                            out[(int64_t)b * p.ld] = p.scale * ((double)s64 / (double)(eb1 - eb0));
                    }
                }
            } else {
                // ---- wide bins (>= 128 bases): every warp STREAMS a contiguous run of bins -- the
                // bins of a region are one contiguous stretch of coverage -- with 16-byte loads,
                // four 512-byte rows in flight per warp.  A row (128 bases) meets at most one
                // bin edge: the lanes keep a running partial sum for the current bin and one for
                // the bin after the edge, and the warp reduces once per BIN, not per row.
                const int per = (n + BWARPS - 1) / BWARPS;
                const int i0 = warp * per, i1 = min(n, i0 + per);
                if (i0 < i1) {
                    const int lo = edge(i0), hi = edge(i1);
                    int k = i0, nxt = edge(i0 + 1);
                    S acc = 0;
                    constexpr int UW = ROWS_IN_FLIGHT<ST>;
                    for (int q0 = lo & ~3; q0 < hi; q0 += 128 * UW) {
                        Raw4<ST> x[UW];
#pragma unroll
                        for (int u = 0; u < UW; u++) {
                            const int q = q0 + u * 128 + lane * 4;
                            x[u] = Raw4<ST>{};
                            if (q < hi) x[u] = load4_cs(src + q);
                        }
#pragma unroll
                        for (int u = 0; u < UW; u++) {
                            const int row = q0 + u * 128;
                            if (row >= hi) break;
                            const int q = row + lane * 4;
                            const int4 xu = widen4(x[u]);
                            auto a0 = word_val<V>(xu.x), a1 = word_val<V>(xu.y), a2 = word_val<V>(xu.z),
                                 a3 = word_val<V>(xu.w);
                            if (row < lo || row + 128 > hi) {           // first / last row of the run
                                a0 = (q >= lo && q < hi) ? a0 : 0;
                                a1 = (q + 1 >= lo && q + 1 < hi) ? a1 : 0;
                                a2 = (q + 2 >= lo && q + 2 < hi) ? a2 : 0;
                                a3 = (q + 3 >= lo && q + 3 < hi) ? a3 : 0;
                            }
                            const S tot = ((S)a0 + a1) + ((S)a2 + a3);
                            if (row + 128 >= nxt) {                     // this row ends the current bin
                                const int c = nxt - q;                  // this lane's elements before the edge
                                const S before = (S)(c > 0 ? a0 : 0) + (c > 1 ? a1 : 0) +
                                                 (c > 2 ? a2 : 0) + (c > 3 ? a3 : 0);
                                S t = acc + before;
#pragma unroll
                                for (int dd = 16; dd > 0; dd >>= 1) t += __shfl_xor_sync(0xffffffffu, t, dd);
                                const int b0 = edge(k);
                                if (lane == 0) out[(int64_t)k * p.ld] = p.scale * ((double)t / (double)(nxt - b0));
                                acc = after_edge<V>(tot, before, c, a0, a1, a2, a3);
                                k++;
                                nxt = k < i1 ? edge(k + 1) : 0x7fffffff;
                            } else {
                                acc += tot;
                            }
                        }
                    }
                }
            }
        }
        r += step;
        if (r >= R) break;
        __syncthreads();                    // edges, wcount, the ring slot and the buffer are reused
    }
    // the copy issued for the (non-existent) region after the last one carries no bytes
}

template <class V>
__global__ void __launch_bounds__(BT)
bin_mean_kernel(BinArgs p, const BinDesc* __restrict__ desc, int64_t R, int buf_ints, int nbuf) {
    __shared__ MeanSmem sm;
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return bin_mean_run<V, uint16_t>(p, desc, R, buf_ints, nbuf, sm);
    }
    bin_mean_run<V, int32_t>(p, desc, R, buf_ints, nbuf, sm);
}

// ---- long regions with wide bins: runs of WIDE_RUN bins of all such regions in one pool --------
// One warp STREAMS a run of consecutive bins -- one contiguous stretch of coverage -- with
// 16-byte loads, four 512-byte rows in flight.  A row (128 bases) meets at most one bin edge
// (bins are >= 128 wide): the lanes keep a partial sum for the current bin, the warp reduces
// once per bin.  Bin i has bsz + [rank[i] <= dif] elements (util.R:74-80).
constexpr int WIDE_RUN = 16;

template <class V, class ST>
__device__ __forceinline__ void bin_wide_run(const BinArgs& p, const BinDesc* __restrict__ desc,
                                             const int32_t* __restrict__ long_list,
                                             unsigned int* __restrict__ long_count) {
    using S = typename Val<V>::Sum;
    const int lane = threadIdx.x & 31;
    const int n = p.n;
    const int runs = (n + WIDE_RUN - 1) / WIDE_RUN;
    const int64_t units = (int64_t)(*long_count) * runs;
    if (units == 0) return;                 // no such region: not a single atomic
    // units are handed out by a counter (long_count[1]): gene lengths are heavy-tailed, and a fixed
    // stride would leave the kernel waiting for the warp that drew the longest regions
    for (;;) {
        unsigned long long u = 0;
        if (lane == 0) u = atomicAdd(reinterpret_cast<unsigned long long*>(long_count + 2), 1ull);
        u = __shfl_sync(0xffffffffu, u, 0);
        if ((int64_t)u >= units) break;
        const int64_t r = long_list[u / runs];
        const int i0 = (int)(u % runs) * WIDE_RUN, i1 = min(n, i0 + WIDE_RUN);
        const BinDesc d = load_bin_desc(desc + r);
        const int bsz = d.bsz, dif = d.dif;
        // lane l knows whether bin i0 + l is one base wider; the start of bin i0 needs the count before it
        int pre = 0;
        unsigned extra = 0;
        if (dif > 0) {
            for (int j = lane; j < i0; j += 32) pre += (__ldg(p.rank + j) <= dif);
#pragma unroll
            for (int dd = 16; dd > 0; dd >>= 1) pre += __shfl_xor_sync(0xffffffffu, pre, dd);
            extra = __ballot_sync(0xffffffffu, i0 + lane < i1 && __ldg(p.rank + i0 + lane) <= dif);
        }
        const int lo = d.a + i0 * bsz + pre;
        const int hi = lo + (i1 - i0) * bsz + __popc(extra);
        const ST* src = reinterpret_cast<const ST*>(p.cov) + (int64_t)(((uint64_t)(uint32_t)d.off_hi << 32) | (uint32_t)d.off_lo);
        double* out = p.out + r;
        int k = i0, b0 = lo, nxt = lo + bsz + (int)(extra & 1u);
        S acc = 0;
        constexpr int UW = ROWS_IN_FLIGHT<ST>;
        // the rows of the NEXT trip are requested before this trip's rows are summed
        auto fetch = [&](int q0, Raw4<ST>* x) {
#pragma unroll
            for (int v = 0; v < UW; v++) {
                const int q = q0 + v * 128 + lane * 4;
                x[v] = Raw4<ST>{};
                if (q < hi) x[v] = load4_cs(src + q);
            }
        };
        Raw4<ST> x[UW], y[UW];
        fetch(lo & ~3, x);
        for (int q0 = lo & ~3; q0 < hi; q0 += 128 * UW) {
            if (q0 + 128 * UW < hi) fetch(q0 + 128 * UW, y);
#pragma unroll
            for (int v = 0; v < UW; v++) {
                const int row = q0 + v * 128;
                if (row >= hi) break;
                const int q = row + lane * 4;
                const int4 xv = widen4(x[v]);
                auto a0 = word_val<V>(xv.x), a1 = word_val<V>(xv.y), a2 = word_val<V>(xv.z),
                     a3 = word_val<V>(xv.w);
                if (row < lo || row + 128 > hi) {           // first / last row of the run
                    a0 = (q >= lo && q < hi) ? a0 : 0;
                    a1 = (q + 1 >= lo && q + 1 < hi) ? a1 : 0;
                    a2 = (q + 2 >= lo && q + 2 < hi) ? a2 : 0;
                    a3 = (q + 3 >= lo && q + 3 < hi) ? a3 : 0;
                }
                const S tot = ((S)a0 + a1) + ((S)a2 + a3);
                if (row + 128 >= nxt) {                     // this row ends the current bin
                    const int c = nxt - q;                  // this lane's elements before the edge
                    const S before = (S)(c > 0 ? a0 : 0) + (c > 1 ? a1 : 0) +
                                     (c > 2 ? a2 : 0) + (c > 3 ? a3 : 0);
                    S t = acc + before;
#pragma unroll
                    for (int dd = 16; dd > 0; dd >>= 1) t += __shfl_xor_sync(0xffffffffu, t, dd);
                    if (lane == 0) out[(int64_t)k * p.ld] = p.scale * ((double)t / (double)(nxt - b0));
                    acc = after_edge<V>(tot, before, c, a0, a1, a2, a3);
                    k++;
                    b0 = nxt;
                    nxt = k < i1 ? nxt + bsz + (int)((extra >> (k - i0)) & 1u) : 0x7fffffff;
                } else {
                    acc += tot;
                }
            }
#pragma unroll
            for (int v = 0; v < UW; v++) x[v] = y[v];
        }
    }
}

template <class V>
__global__ void __launch_bounds__(BT, 3)
bin_wide_kernel(BinArgs p, const BinDesc* __restrict__ desc, const int32_t* __restrict__ long_list,
                unsigned int* __restrict__ long_count) {
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return bin_wide_run<V, uint16_t>(p, desc, long_list, long_count);
    }
    bin_wide_run<V, int32_t>(p, desc, long_list, long_count);
}

// ---- interpolation of short segments (util.R:17-73) ------------------------------------------
struct InterpArgs {
    const int32_t* cov;
    const unsigned long long* bound;
    const int64_t* off;
    const int32_t* len;
    int where, f1, f2, n;
    int interp, seed, sample_kind;
    double scale;
    double* out;
    int64_t ld;
    const int32_t* short_list;
    const unsigned int* short_count;
};

// dynamic smem per warp-CTA: 4n doubles + 2n ints + RRng
template <class V, class ST>
__device__ __forceinline__ void interp_run(const InterpArgs& p) {
    using E = typename std::conditional<sizeof(ST) == 2, uint16_t, V>::type;     // an element as stored
    extern __shared__ double shd[];
    const int n = p.n;
    double* y = shd;               // input values (L) / neighbourhood vector (n)
    double* cb = shd + n;          // spline b / neighbourhood pre-fill copy
    double* cc = shd + 2 * n;
    double* cd = shd + 3 * n;
    int* ia = reinterpret_cast<int*>(shd + 4 * n);   // n ints
    int* ib = ia + n;                                 // n ints
    RRng* rng = reinterpret_cast<RRng*>(ib + n);
    const int lane = threadIdx.x;
    const unsigned int count = *p.short_count;
    for (unsigned int w = blockIdx.x; w < count; w += gridDim.x) {
        const int64_t r = p.short_list[w];
        const int L_all = p.len[r];
        const Seg sg = segment_of(L_all, p.where, p.f1, p.f2);
        const int L = sg.b - sg.a;
        const E* src = reinterpret_cast<const E*>(p.cov) + p.off[r] + sg.a;
        double* out = p.out + r;
        __syncwarp();
        bool neighborhood = p.interp == RCP_INTERP_NEIGHBORHOOD;
        if (p.interp == RCP_INTERP_AUTO) neighborhood = ((double)(n - L) / (double)n) < 0.2;
        if (neighborhood && (L < 4 || n < 6)) {
            // R's sample() would stop(); flagged as NaN row (the host rejects these sizes first)
            for (int i = lane; i < n; i += 32) out[(int64_t)i * p.ld] = nan("");
            continue;
        }
        if (!neighborhood) {
            // ---- stats::spline(method = "fmm"), x = 1..L, xout = seq(1, L, length.out = n)
            for (int i = lane; i < L; i += 32) y[i] = (double)src[i];
            __syncwarp();
            if (lane == 0) {
                double *b = cb, *c = cc, *d = cd;
                for (int i = 0; i < L; i++) b[i] = c[i] = d[i] = 0.0;
                if (L == 2) {
                    b[0] = b[1] = y[1] - y[0];
                } else if (L >= 3) {
                    const int nm1 = L - 1;
                    d[0] = 1.0;                       // x[i+1] - x[i] == 1
                    c[1] = (y[1] - y[0]) / d[0];
                    for (int i = 1; i < nm1; i++) {
                        d[i] = 1.0;
                        b[i] = 2.0 * (d[i - 1] + d[i]);
                        c[i + 1] = (y[i + 1] - y[i]) / d[i];
                        c[i] = c[i + 1] - c[i];
                    }
                    b[0] = -d[0];
                    b[L - 1] = -d[L - 2];
                    c[0] = c[L - 1] = 0.0;
                    if (L > 3) {
                        c[0] = c[2] / 2.0 - c[1] / 2.0;              // x[3]-x[1] = x[2]-x[0] = 2
                        c[L - 1] = c[L - 2] / 2.0 - c[L - 3] / 2.0;
                        c[0] = c[0] * d[0] * d[0] / 3.0;             // x[3]-x[0] = 3
                        c[L - 1] = -c[L - 1] * d[L - 2] * d[L - 2] / 3.0;
                    }
                    for (int i = 1; i < L; i++) {
                        const double t = d[i - 1] / b[i - 1];
                        b[i] = b[i] - t * d[i - 1];
                        c[i] = c[i] - t * c[i - 1];
                    }
                    c[L - 1] = c[L - 1] / b[L - 1];
                    for (int i = L - 2; i >= 0; i--) c[i] = (c[i] - d[i] * c[i + 1]) / b[i];
                    b[L - 1] = (y[L - 1] - y[L - 2]) / d[L - 2] + d[L - 2] * (c[L - 2] + 2.0 * c[L - 1]);
                    for (int i = 0; i < nm1; i++) {
                        b[i] = (y[i + 1] - y[i]) / d[i] - d[i] * (c[i + 1] + 2.0 * c[i]);
                        d[i] = (c[i + 1] - c[i]) / d[i];
                        c[i] = 3.0 * c[i];
                    }
                    c[L - 1] = 3.0 * c[L - 1];
                    d[L - 1] = d[L - 2];
                }
            }
            __syncwarp();
            const double by = n > 2 ? ((double)L - 1.0) / (double)(n - 1) : 0.0;
            for (int l = lane; l < n; l += 32) {
                double ul = 1.0 + (double)l * by;
                if (l == 0) ul = 1.0;
                if (l == n - 1 && n > 1) ul = (double)L;
                int i = (int)floor(ul) - 1;
                if (i > L - 2) i = L - 2;
                if (i < 0) i = 0;
                const double dx = ul - (double)(i + 1);
                double v = y[i] + dx * (cb[i] + dx * (cc[i] + dx * cd[i]));
                if (v < 0.0) v = 0.0;                                 // util.R:42,47
                out[(int64_t)l * p.ld] = p.scale * v;
            }
        } else {
            // ---- neighbourhood fill (util.R:24-38 / 54-68)
            for (int i = lane; i < n; i += 32) {
                y[i] = nan("");
                ia[i] = 0;
            }
            __syncwarp();
            if (lane == 0) {
                y[0] = (double)src[0];
                y[1] = (double)src[1];
                y[n - 2] = (double)src[L - 2];
                y[n - 1] = (double)src[L - 1];
                rng->seed((uint32_t)p.seed, p.sample_kind);
                // orig.pos <- sort(sample(3:(n-2), L-4)): mark the picks, sweep in order
                const int pool = n - 4, k = L - 4;
                int* x = ib;
                for (int i = 0; i < pool; i++) x[i] = i;
                int m = pool;
                for (int i = 0; i < k; i++) {
                    const int j = (int)rng->index((uint32_t)m);
                    ia[x[j]] = 1;                      // value 3 + x[j]  (1-based position)
                    x[j] = x[--m];
                }
                int q = 2;
                for (int i = 0; i < pool; i++)
                    if (ia[i]) y[2 + i] = (double)src[q++];
            }
            __syncwarp();
            for (int i = lane; i < n; i += 32) cb[i] = y[i];
            __syncwarp();
            for (int z = lane; z < n; z += 32) {
                double v = cb[z];
                if (isnan(v)) {                        // mean(y[c(z-2,z-1,z+1,z+2)], na.rm=TRUE)
                    double s = 0.0;
                    int c = 0;
                    const int nb[4] = {z - 2, z - 1, z + 1, z + 2};
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        const double u = cb[nb[t]];    // z in [2, n-3] -> always in range
                        if (!isnan(u)) { s += u; c++; }
                    }
                    v = c ? s / (double)c : nan("");
                }
                out[(int64_t)z * p.ld] = p.scale * v;
            }
        }
    }
}

template <class V>
__global__ void __launch_bounds__(32) interp_kernel(InterpArgs p) {
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return interp_run<V, uint16_t>(p);
    }
    interp_run<V, int32_t>(p);
}

// ---- per-base matrix --------------------------------------------------------------------------
struct BaseArgs {
    const int32_t* cov;
    const unsigned long long* bound;
    const int64_t* off;
    const int32_t* len;
    const uint8_t* is_null;
    int where, f1, f2;
    int64_t R, n_cols;
    double scale;
    double* out;
    int64_t ld;
};

struct BaseSmem {
    int tile[32][33];
    int64_t r_off[32];
    int r_a[32], r_b[32];
};
template <class V, class S>
__device__ __forceinline__ void base_matrix_run(const BaseArgs& p, BaseSmem& sm) {
    auto& tile = sm.tile;
    auto& r_off = sm.r_off;
    auto& r_a = sm.r_a;
    auto& r_b = sm.r_b;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t r0 = (int64_t)blockIdx.y * 32, k0 = (int64_t)blockIdx.x * 32;
    if (ty == 0) {
        const int64_t r = r0 + tx;
        int a = 0, b = 0;
        int64_t o = 0;
        if (r < p.R && !p.is_null[r]) {
            const Seg sg = segment_of(p.len[r], p.where, p.f1, p.f2);
            a = sg.a;
            b = sg.b;
            o = p.off[r];
        }
        r_off[tx] = o;
        r_a[tx] = a;
        r_b[tx] = b;
    }
    __syncthreads();
    for (int jj = ty; jj < 32; jj += 8) {
        const int64_t k = k0 + tx;
        const int q = r_a[jj] + (int)k;
        int v = 0;
        if (k < p.n_cols && q < r_b[jj]) v = __ldg(reinterpret_cast<const S*>(p.cov) + r_off[jj] + q);
        tile[jj][tx] = v;
    }
    __syncthreads();
    for (int jj = ty; jj < 32; jj += 8) {
        const int64_t k = k0 + jj, r = r0 + tx;
        if (r < p.R && k < p.n_cols) p.out[k * p.ld + r] = p.scale * word_double<V>(tile[tx][jj]);
    }
}

template <class V>
__global__ void __launch_bounds__(256) base_matrix_kernel(BaseArgs p) {
    __shared__ BaseSmem sm;
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return base_matrix_run<V, uint16_t>(p, sm);
    }
    base_matrix_run<V, int32_t>(p, sm);
}

// Wide-tile version of the same transpose: 32 regions x 256 columns per CTA.  Rows are read with
// 16-byte loads when the segment start is 4-aligned (always for whole windows), columns leave as
// 256-byte runs of 32 consecutive regions, two doubles per lane when the output allows 16-byte
// stores.  The tile index runs along x (linear, no 65535 limit).
constexpr int BW_ROWS = 32, BW_COLS = 256;

struct BaseWideSmem {
    int tile[BW_ROWS][BW_COLS + 1];
    int64_t r_off[BW_ROWS];
    int r_a[BW_ROWS], r_b[BW_ROWS];
};
template <class V, class S>
__device__ __forceinline__ void base_matrix_wide_run(const BaseArgs& p, int64_t col_tiles, int vec_store,
                                                     BaseWideSmem& sm) {
    auto& tile = sm.tile;
    auto& r_off = sm.r_off;
    auto& r_a = sm.r_a;
    auto& r_b = sm.r_b;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r0 = ((int64_t)blockIdx.x / col_tiles) * BW_ROWS;
    const int64_t k0 = ((int64_t)blockIdx.x % col_tiles) * BW_COLS;
    if (tid < BW_ROWS) {
        const int64_t r = r0 + tid;
        int a = 0, b = 0;
        int64_t o = 0;
        if (r < p.R && !p.is_null[r]) {
            const Seg sg = segment_of(p.len[r], p.where, p.f1, p.f2);
            a = sg.a;
            b = sg.b;
            o = p.off[r];
        }
        r_off[tid] = o;
        r_a[tid] = a;
        r_b[tid] = b;
    }
    __syncthreads();
    for (int jj = warp; jj < BW_ROWS; jj += 8) {
        const int a = r_a[jj], b = r_b[jj];
        const S* src = reinterpret_cast<const S*>(p.cov) + r_off[jj] + a + k0;       // column k0 of this region
        const int avail = (int)min((int64_t)(b - a) - k0, (int64_t)BW_COLS);   // columns with data
#pragma unroll
        for (int h = 0; h < BW_COLS / 128; h++) {
            const int c = h * 128 + lane * 4;
            int4 v = make_int4(0, 0, 0, 0);
            if ((a & 3) == 0 && c + 3 < avail) {
                v = load4_g(src + c);
            } else {
                if (c < avail) v.x = __ldg(src + c);
                if (c + 1 < avail) v.y = __ldg(src + c + 1);
                if (c + 2 < avail) v.z = __ldg(src + c + 2);
                if (c + 3 < avail) v.w = __ldg(src + c + 3);
            }
            tile[jj][c] = v.x;
            tile[jj][c + 1] = v.y;
            tile[jj][c + 2] = v.z;
            tile[jj][c + 3] = v.w;
        }
    }
    __syncthreads();
    const int ncol = (int)min((int64_t)BW_COLS, p.n_cols - k0);
    if (vec_store && r0 + BW_ROWS <= p.R) {
        // lanes 0..15 write column c, lanes 16..31 column c + 1; each lane two regions (16 bytes)
        const int rr = (lane & 15) * 2, dc = lane >> 4;
        for (int c = warp * 2 + dc; c < ncol; c += 16) {
            const double2 v = make_double2(p.scale * word_double<V>(tile[rr][c]), p.scale * word_double<V>(tile[rr + 1][c]));
            *reinterpret_cast<double2*>(p.out + (k0 + c) * p.ld + r0 + rr) = v;
        }
    } else {
        const int64_t r = r0 + lane;
        if (r < p.R)
            for (int c = warp; c < ncol; c += 8) p.out[(k0 + c) * p.ld + r] = p.scale * word_double<V>(tile[lane][c]);
    }
}

template <class V>
__global__ void __launch_bounds__(256) base_matrix_wide_kernel(BaseArgs p, int64_t col_tiles, int vec_store) {
    __shared__ BaseWideSmem sm;
    if constexpr (std::is_same<V, int32_t>::value) {
        if (cov_narrow(p.bound)) return base_matrix_wide_run<V, uint16_t>(p, col_tiles, vec_store, sm);
    }
    base_matrix_wide_run<V, int32_t>(p, col_tiles, vec_store, sm);
}

template <class V>
int bin_matrix_impl(const Coverage& cv, int where, int f1, int f2, int n_bins, int stat,
                    int interp, int seed, int sample_kind, double* d_out, int64_t ld) {
    const int64_t R = cv.n_regions;
    if (R == 0) return RCP_OK;
    // rank table of `set.seed(seed); sample(1:n, n)` (host, n is small)
    std::vector<int> rank((size_t)n_bins), perm((size_t)n_bins), scratch((size_t)n_bins);
    {
        RRng* rng = new RRng;
        rng->seed((uint32_t)seed, sample_kind);
        rng->sample(n_bins, n_bins, scratch.data(), perm.data());
        delete rng;
        for (int pos = 0; pos < n_bins; pos++) rank[(size_t)perm[(size_t)pos] - 1] = pos + 1;
    }
    int* d_rank = nullptr;
    int32_t* short_list = nullptr;
    unsigned int* short_count = nullptr;
    BinDesc* d_desc = nullptr;
    int32_t* long_list = nullptr;
    unsigned int* long_count = nullptr;
    struct Release {            // every exit, error returns included, frees the scratch buffers
        int** rank;
        int32_t** shorts;
        unsigned int** short_n;
        BinDesc** desc;
        int32_t** longs;
        unsigned int** long_n;
        ~Release() {
            dfree(*desc);
            dfree(*longs);
            dfree(*long_n);
            dfree(*rank);
            dfree(*shorts);
            dfree(*short_n);
        }
    } release{&d_rank, &short_list, &short_count, &d_desc, &long_list, &long_count};
    RCP_TRY(dalloc(&d_rank, (size_t)n_bins));
    RCP_TRY(dalloc(&short_list, (size_t)R));
    RCP_TRY(dalloc(&short_count, 1));
    RCP_CUDA(cudaMemcpyAsync(d_rank, rank.data(), (size_t)n_bins * sizeof(int),
                             cudaMemcpyHostToDevice, g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(short_count, 0, sizeof(unsigned int), g_ctx.stream));
    // the pageable source of the rank copy must outlive the copy: cudaMemcpyAsync from pageable
    // memory returns after the source has been staged, so `rank` may go out of scope later.
    BinArgs a;
    a.cov = cv.cov;
    a.bound = cv.d_bound;
    a.off = cv.off;
    a.len = cv.len;
    a.is_null = cv.is_null;
    a.rank = d_rank;
    a.where = where;
    a.f1 = f1;
    a.f2 = f2;
    a.n = n_bins;
    a.scale = cv.scale;
    a.out = d_out;
    a.ld = ld;
    a.short_list = short_list;
    a.short_count = short_count;
    const size_t edge_bytes = (((size_t)n_bins + 1 + 3) & ~(size_t)3) * sizeof(int);
    if (edge_bytes > 150 * 1024) return fail(RCP_ERR_UNSUPPORTED, "more than 38399 bins per segment");
    if (stat == RCP_STAT_MEDIAN) {
        StageTimer t(ST_PROF_BIN);
        const size_t smem = edge_bytes;
        if (smem > 48 * 1024)
            RCP_CUDA(cudaFuncSetAttribute(bin_median_kernel<V>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bin_median_kernel<V><<<(unsigned)R, CTA, smem, g_ctx.stream>>>(a);
        RCP_LAUNCHED();
    } else {
        // two staging buffers per CTA; the kernel is persistent (one resident wave of CTAs)
        RCP_TRY(dalloc(&d_desc, (size_t)R));
        StageTimer t(ST_PROF_BIN);
        // longest segment any region can have here, + alignment slack, capped at one staged run
        int64_t seg_max = cv.max_len;
        if (where == RCP_WHERE_UPSTREAM) seg_max = std::min<int64_t>(seg_max, f1);
        else if (where == RCP_WHERE_DOWNSTREAM) seg_max = std::min<int64_t>(seg_max, f2);
        else if (where == RCP_WHERE_CENTER) seg_max = std::max<int64_t>(seg_max - f1 - f2, 0);
        // (+ 8 more: a narrow coverage stages from an 8-aligned base into half a buffer)
        int buf_ints = (int)std::min<int64_t>(STAGE_INTS, ((seg_max + 18) & ~(int64_t)3));
        // CTAs per SM: four, unless the typical bin is wide (mean segment / bins >= 128 bases:
        // gene bodies).  Wide bins are summed straight from global memory by one warp each and
        // are bound by the loads in flight, so they want all 64 warps of the SM; the staging
        // buffers (used by the shorter regions only) shrink to make room.
        int per_sm = 4;
        {
            const int64_t live = std::max<int64_t>(R - cv.n_null, 1);
            int64_t seg_mean = cv.total_len / live;
            if (where == RCP_WHERE_UPSTREAM) seg_mean = std::min<int64_t>(seg_mean, f1);
            else if (where == RCP_WHERE_DOWNSTREAM) seg_mean = std::min<int64_t>(seg_mean, f2);
            else if (where == RCP_WHERE_CENTER) seg_mean = std::max<int64_t>(seg_mean - f1 - f2, 0);
            if (seg_mean / n_bins >= 128) {
                per_sm = 8;
                buf_ints = std::min(buf_ints, 6144);
            }
        }
        RCP_TRY(dalloc(&long_list, (size_t)R));
        RCP_TRY(dalloc(&long_count, 4));        // [0] regions in the list, [2..3] unit counter of bin_wide_kernel
        RCP_CUDA(cudaMemsetAsync(long_count, 0, 4 * sizeof(unsigned int), g_ctx.stream));
        bin_desc_kernel<<<(unsigned)((R + CTA - 1) / CTA), CTA, 0, g_ctx.stream>>>(
            R, cv.off, cv.len, cv.is_null, where, f1, f2, n_bins, buf_ints, d_desc, long_list, long_count,
            cv.d_bound);
        RCP_LAUNCHED();
        // CTAs per SM and buffers per CTA: as much shared memory as possible in flight
        if (const char* e = getenv("RCP_BIN_CTAS")) per_sm = std::max(1, atoi(e));     // tuning
        // the edges of many bins leave no room for a staging buffer at this many CTAs per SM:
        // fewer CTAs (150 KB of edges and one 48 KB buffer fit one CTA)
        const int64_t buf_bytes = (int64_t)buf_ints * (int64_t)sizeof(int);
        auto budget_at = [](int k) { return (int64_t)(220 * 1024 / k) - 1024; };
        while (per_sm > 1 && budget_at(per_sm) - (int64_t)edge_bytes < buf_bytes) per_sm--;
        const int64_t room = budget_at(per_sm) - (int64_t)edge_bytes;
        if (room < buf_bytes)
            return fail(RCP_ERR_UNSUPPORTED, "bin kernel does not fit (%zu bytes of bin edges)", edge_bytes);
        const int nbuf = (int)std::min<int64_t>(room / buf_bytes, NBUF_MAX);
        const size_t smem = edge_bytes + (size_t)nbuf * buf_ints * sizeof(int);
        RCP_CUDA(cudaFuncSetAttribute(bin_mean_kernel<V>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
        int fit = 0;
        RCP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, bin_mean_kernel<V>, BT, smem));
        if (fit < 1) return fail(RCP_ERR_UNSUPPORTED, "bin kernel does not fit (%zu bytes of shared memory)", smem);
        const int64_t grid = std::min<int64_t>(R, (int64_t)g_ctx.sm_count * std::min(fit, per_sm));
        bin_mean_kernel<V><<<(unsigned)grid, BT, smem, g_ctx.stream>>>(a, d_desc, R, buf_ints, nbuf);
        RCP_LAUNCHED();
        // (nothing to do when no region is long: the warps find zero units)
        bin_wide_kernel<V><<<(unsigned)(g_ctx.sm_count * 8), BT, 0, g_ctx.stream>>>(a, d_desc, long_list, long_count);
        RCP_LAUNCHED();
    }
    InterpArgs ia;
    ia.cov = cv.cov;
    ia.bound = cv.d_bound;
    ia.off = cv.off;
    ia.len = cv.len;
    ia.where = where;
    ia.f1 = f1;
    ia.f2 = f2;
    ia.n = n_bins;
    ia.interp = interp;
    ia.seed = seed;
    ia.sample_kind = sample_kind;
    ia.scale = cv.scale;
    ia.out = d_out;
    ia.ld = ld;
    ia.short_list = short_list;
    ia.short_count = short_count;
    const size_t ismem = (size_t)n_bins * (4 * sizeof(double) + 2 * sizeof(int)) + 8 + sizeof(RRng);
    if (ismem > 220 * 1024) {
        // more bins than the interpolation kernel can hold: fine as long as no segment is shorter
        // than the bin count.  The bin kernels have listed those; one read-back tells.
        unsigned int n_short = 0;
        RCP_CUDA(cudaMemcpyAsync(&n_short, short_count, sizeof(unsigned int), cudaMemcpyDeviceToHost,
                                 g_ctx.stream));
        RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        if (n_short == 0) return RCP_OK;
        return fail(RCP_ERR_UNSUPPORTED,
                    "%u segments are shorter than the %d bins; interpolation supports at most %d bins",
                    n_short, n_bins, (int)((220 * 1024 - 8 - sizeof(RRng)) / (4 * sizeof(double) + 2 * sizeof(int))));
    }
    if (ismem > 48 * 1024)
        RCP_CUDA(cudaFuncSetAttribute(interp_kernel<V>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)ismem));
    int iblocks = g_ctx.sm_count * 8;
    if ((int64_t)iblocks > R) iblocks = (int)R;
    {
        StageTimer t(ST_PROF_INTERP);
        interp_kernel<V><<<(unsigned)iblocks, 32, ismem, g_ctx.stream>>>(ia);
        RCP_LAUNCHED();
    }
    return RCP_OK;
}

template <class V>
int base_matrix_impl(const Coverage& cv, int where, int f1, int f2, int64_t n_cols,
                     double* d_out, int64_t ld) {
    const int64_t R = cv.n_regions;
    if (R == 0 || n_cols == 0) return RCP_OK;
    BaseArgs a;
    a.cov = cv.cov;
    a.bound = cv.d_bound;
    a.off = cv.off;
    a.len = cv.len;
    a.is_null = cv.is_null;
    a.where = where;
    a.f1 = f1;
    a.f2 = f2;
    a.R = R;
    a.n_cols = n_cols;
    a.scale = cv.scale;
    a.out = d_out;
    a.ld = ld;
    StageTimer t(ST_PROF_BASE);
    if (n_cols >= 128) {
        // wide tiles; 16-byte stores need an even leading dimension and a 16-byte aligned matrix
        const int64_t col_tiles = (n_cols + BW_COLS - 1) / BW_COLS, row_tiles = (R + BW_ROWS - 1) / BW_ROWS;
        if (col_tiles * row_tiles <= 0x7fffffff) {
            const int vec = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(d_out) & 15u) == 0);
            base_matrix_wide_kernel<V><<<(unsigned)(col_tiles * row_tiles), 256, 0, g_ctx.stream>>>(
                a, col_tiles, vec);
            RCP_LAUNCHED();
            return RCP_OK;
        }
    }
    const int64_t gy = (R + 31) / 32, gx = (n_cols + 31) / 32;
    if (gy > 65535) {
        // grid.y is limited to 65535: walk the rows in slabs
        for (int64_t y0 = 0; y0 < gy; y0 += 65535) {
            BaseArgs s = a;
            const int64_t rows0 = y0 * 32;
            s.off = a.off + rows0;
            s.len = a.len + rows0;
            s.is_null = a.is_null + rows0;
            s.R = (R - rows0) < 65535 * 32 ? (R - rows0) : 65535 * 32;
            s.out = a.out + rows0;
            const int64_t gys = (s.R + 31) / 32;
            base_matrix_kernel<V><<<dim3((unsigned)gx, (unsigned)gys), dim3(32, 8), 0, g_ctx.stream>>>(s);
            RCP_LAUNCHED();
        }
    } else {
        base_matrix_kernel<V><<<dim3((unsigned)gx, (unsigned)gy), dim3(32, 8), 0, g_ctx.stream>>>(a);
        RCP_LAUNCHED();
    }
    return RCP_OK;
}

}  // namespace

// out points to DEVICE memory here; the api layer stages host outputs.
int bin_matrix_device(const Coverage& cv, int where, int f1, int f2, int n_bins, int stat,
                      int interp, int seed, int sample_kind, double* d_out, int64_t ld) {
    if (cv.value_type == RCP_VALUE_FLOAT32)
        return bin_matrix_impl<float>(cv, where, f1, f2, n_bins, stat, interp, seed, sample_kind, d_out, ld);
    return bin_matrix_impl<int32_t>(cv, where, f1, f2, n_bins, stat, interp, seed, sample_kind, d_out, ld);
}

int base_matrix_device(const Coverage& cv, int where, int f1, int f2, int64_t n_cols,
                       double* d_out, int64_t ld) {
    if (cv.value_type == RCP_VALUE_FLOAT32) return base_matrix_impl<float>(cv, where, f1, f2, n_cols, d_out, ld);
    return base_matrix_impl<int32_t>(cv, where, f1, f2, n_cols, d_out, ld);
}

}  // namespace rcp
