// rcp_reads_load: reads -> device index.
//
// Every read is mapped to a 32-bit GLOBAL coordinate  g = chrom_off[chrom] + pos  (chromosomes
// laid end to end with a 2-position gap), and two arrays are sorted INDEPENDENTLY:
//     xs = sorted(global start)          ye = sorted(global end + 1)
// Exact coverage then follows from ranks alone:
//     cov(p) = #{xs <= p} - #{ye <= p}
// so the coverage kernels never need (start,end) pairs, never depend on the read width and can
// cut any region into tiles without carrying state between tiles (coverage.cu).
// Replaces splitBySeqname + the per-region findOverlaps/coverage of the reference
// (/root/reference/R/util.R:1-13, R/coverage.R:189-201).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "rcp_internal.cuh"

namespace rcp {

namespace {

constexpr int TPB = 256;

// Reads -> global coordinates.  err bits: 1 chrom id out of range, 2 start < 1 or end < start,
// 4 start beyond the chromosome.
struct ExcBuf {
    uint32_t* xw;        // start + w of reads whose width differs from w ("assumed" end + 1)
    uint32_t* e1;        // their true end + 1
    int8_t* st;          // their strand
    uint32_t cap;
    unsigned int* count; // may exceed cap: overflow => uniform-width mode is abandoned
    uint32_t* w_out;     // the candidate width used
};

__device__ __forceinline__ bool map_read(int c, int64_t s, int64_t e, int st, int n_chrom,
                                         const uint32_t* __restrict__ chrom_off,
                                         const int64_t* __restrict__ chrom_len, int frag_len,
                                         uint32_t* gs, uint32_t* ge1, unsigned int* err) {
    if (c < 0 || c >= n_chrom) { *err |= 1u; return false; }
    if (s < 1 || e < s) { *err |= 2u; return false; }
    const int64_t len = chrom_len[c];
    if (frag_len > 0) {           // resize(fix="start"): '-' keeps its end
        if (st < 0) s = e - frag_len + 1;
        else e = s + frag_len - 1;
    }
    if (s < 1) s = 1;             // trim()
    if (e > len) e = len;
    if (s > len || e < s) { *err |= 4u; return false; }
    *gs = chrom_off[c] + (uint32_t)s;
    *ge1 = chrom_off[c] + (uint32_t)e + 1u;
    return true;
}

// NA seqlengths: the largest read end per chromosome, fragment extension applied, nothing trimmed
// (chromosomes of unknown length have no end to trim at).  Invalid reads are left to the map kernel.
__global__ void __launch_bounds__(TPB)
chrom_max_end_kernel(int64_t n, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
                     const int32_t* __restrict__ end, const int8_t* __restrict__ strand, int n_chrom,
                     int frag_len, int fixed_width, unsigned long long* __restrict__ max_end) {
    const int64_t stride = (int64_t)gridDim.x * TPB;
    int last_c = -1;
    long long best = 0;
    for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += stride) {
        const int c = chrom[i];
        if (c < 0 || c >= n_chrom) continue;
        const long long s = start[i];
        long long e = end ? (long long)end[i] : s + fixed_width - 1;
        if (frag_len > 0 && !(strand && strand[i] < 0)) e = s + frag_len - 1;
        if (c != last_c) {
            if (last_c >= 0 && best > 0) atomicMax(max_end + last_c, (unsigned long long)best);
            last_c = c;
            best = 0;
        }
        best = max(best, e);
    }
    if (last_c >= 0 && best > 0) atomicMax(max_end + last_c, (unsigned long long)best);
}

// VEC = 4: every thread maps four consecutive reads with 16-byte loads/stores (all arrays
// 16-byte aligned, checked on the host); the n % 4 tail and VEC = 1 use scalar accesses.
template <int VEC, bool HAS_END>
__global__ void __launch_bounds__(TPB)
reads_to_global_kernel(int64_t n, const int32_t* __restrict__ chrom,
                       const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                       const int8_t* __restrict__ strand, const uint32_t* __restrict__ chrom_off,
                       const int64_t* __restrict__ chrom_len, int n_chrom, int frag_len,
                       int fixed_width /* end == nullptr: every read is [start, start + fixed_width - 1] */,
                       uint32_t long_thr /* reads wider than this are counted in exc.count[2] */,
                       uint32_t* __restrict__ g_start, uint32_t* __restrict__ g_end1,
                       uint32_t* __restrict__ xs_out, int8_t* __restrict__ strand_out,
                       unsigned int* __restrict__ err, unsigned long long* __restrict__ cls_count,
                       ExcBuf exc) {
    unsigned int my_err = 0;
    unsigned int np = 0, nm = 0, ns = 0, wmax = 0, nlong = 0;
    bool exc_full = false;
    // candidate common width: the fragment length, else the width of read 0
    uint32_t w = (uint32_t)frag_len;
    if (frag_len <= 0) {
        uint32_t a = 0, b = 0;
        unsigned int e0 = 0;
        if (map_read(chrom[0], start[0], HAS_END ? (int64_t)end[0] : (int64_t)start[0] + fixed_width - 1,
                     strand ? (int)strand[0] : 0, n_chrom, chrom_off,
                     chrom_len, 0, &a, &b, &e0))
            w = b - a;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *exc.w_out = w;

    auto one = [&](int c, int s, int64_t e, int st, uint32_t* gs, uint32_t* ge1) {
        *gs = 0;
        *ge1 = 0;
        if (map_read(c, s, e, st, n_chrom, chrom_off, chrom_len, frag_len, gs, ge1, &my_err)) {
            wmax = max(wmax, *ge1 - *gs);
            nlong += (*ge1 - *gs > long_thr);
            // reads of another width: recorded until the buffer overflows (then uniform-width
            // mode is abandoned anyway and the single counter must not become a hot spot)
            if (*ge1 - *gs != w && !exc_full) {
                // (one look at the counter per thread once it is full: it is a single address)
                if (*reinterpret_cast<volatile unsigned int*>(exc.count) > exc.cap) {
                    exc_full = true;
                } else {
                    const unsigned int k = atomicAdd(exc.count, 1u);
                    if (k < exc.cap) {
                        exc.xw[k] = *gs + w;
                        exc.e1[k] = *ge1;
                        exc.st[k] = (int8_t)(st > 0 ? 1 : (st < 0 ? -1 : 0));
                    }
                }
            }
        }
        np += st > 0;
        nm += st < 0;
        ns += st == 0;
    };
    auto sgn = [](int st) { return (int8_t)(st > 0 ? 1 : (st < 0 ? -1 : 0)); };

    const int64_t stride = (int64_t)gridDim.x * TPB;
    const int64_t n_vec = (VEC == 4) ? (n >> 2) : 0;
    for (int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x; v < n_vec; v += stride) {
        const int4 c4 = __ldg(reinterpret_cast<const int4*>(chrom) + v);
        const int4 s4 = __ldg(reinterpret_cast<const int4*>(start) + v);
        int4 e4 = make_int4(0, 0, 0, 0);
        if (HAS_END) e4 = __ldg(reinterpret_cast<const int4*>(end) + v);
        const int64_t wm1 = (int64_t)fixed_width - 1;
        char4 t4 = make_char4(0, 0, 0, 0);
        if (strand) t4 = __ldg(reinterpret_cast<const char4*>(strand) + v);
        uint4 gs, ge;
        one(c4.x, s4.x, HAS_END ? (int64_t)e4.x : s4.x + wm1, t4.x, &gs.x, &ge.x);
        one(c4.y, s4.y, HAS_END ? (int64_t)e4.y : s4.y + wm1, t4.y, &gs.y, &ge.y);
        one(c4.z, s4.z, HAS_END ? (int64_t)e4.z : s4.z + wm1, t4.z, &gs.z, &ge.z);
        one(c4.w, s4.w, HAS_END ? (int64_t)e4.w : s4.w + wm1, t4.w, &gs.w, &ge.w);
        reinterpret_cast<uint4*>(g_start)[v] = gs;
        reinterpret_cast<uint4*>(g_end1)[v] = ge;
        if (xs_out) reinterpret_cast<uint4*>(xs_out)[v] = gs;
        if (strand_out)
            reinterpret_cast<char4*>(strand_out)[v] = make_char4(sgn(t4.x), sgn(t4.y), sgn(t4.z), sgn(t4.w));
    }
    for (int64_t i = n_vec * 4 + (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += stride) {
        const int st = strand ? (int)strand[i] : 0;
        uint32_t gs, ge1;
        one(chrom[i], start[i], HAS_END ? (int64_t)end[i] : (int64_t)start[i] + fixed_width - 1, st, &gs, &ge1);
        g_start[i] = gs;
        g_end1[i] = ge1;
        if (xs_out) xs_out[i] = gs;
        if (strand_out) strand_out[i] = sgn(st);
    }
    // block-level reduction of the three strand counters and the error mask
    __shared__ unsigned int sh[6];
    if (threadIdx.x < 6) sh[threadIdx.x] = 0;
    __syncthreads();
    for (int d = 16; d > 0; d >>= 1) {
        np += __shfl_xor_sync(0xffffffffu, np, d);
        nm += __shfl_xor_sync(0xffffffffu, nm, d);
        ns += __shfl_xor_sync(0xffffffffu, ns, d);
        my_err |= __shfl_xor_sync(0xffffffffu, my_err, d);
        wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, d));
        nlong += __shfl_xor_sync(0xffffffffu, nlong, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (nlong) atomicAdd(&sh[5], nlong);
        atomicAdd(&sh[0], np);
        atomicAdd(&sh[1], nm);
        atomicAdd(&sh[2], ns);
        atomicOr(&sh[3], my_err);
        atomicMax(&sh[4], wmax);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (sh[0]) atomicAdd(&cls_count[0], (unsigned long long)sh[0]);
        if (sh[1]) atomicAdd(&cls_count[1], (unsigned long long)sh[1]);
        if (sh[2]) atomicAdd(&cls_count[2], (unsigned long long)sh[2]);
        if (sh[3]) atomicOr(err, sh[3]);
        if (sh[4]) atomicMax(&cls_count[3], (unsigned long long)sh[4]);
        if (sh[5]) atomicAdd(exc.count + 2, sh[5]);
    }
}

// correction events of one strand class; slots of other strands become +inf sentinels
__global__ void __launch_bounds__(TPB)
exc_select_kernel(uint32_t n_exc, const uint32_t* __restrict__ xw, const uint32_t* __restrict__ e1,
                  const int8_t* __restrict__ st, int want /* 2 = every strand */,
                  uint32_t* __restrict__ cxs, uint32_t* __restrict__ cye) {
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    if (i >= n_exc) return;
    const bool keep = (want == 2) || ((int)st[i] == want);
    cxs[i] = keep ? xw[i] : 0xffffffffu;
    cye[i] = keep ? e1[i] : 0xffffffffu;
}

// keep the reads of one strand (order is irrelevant: both outputs are sorted afterwards)
__global__ void __launch_bounds__(TPB)
compact_strand_kernel(int64_t n, const uint32_t* __restrict__ g_start,
                      const uint32_t* __restrict__ g_end1, const int8_t* __restrict__ strand,
                      int want, uint32_t* __restrict__ xs, uint32_t* __restrict__ ye /* may be null */,
                      unsigned long long* __restrict__ cursor) {
    const int64_t stride = (int64_t)gridDim.x * TPB;
    const unsigned lane = threadIdx.x & 31;
    const int64_t n_round = (n + 31) & ~(int64_t)31;
    for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n_round; i += stride) {
        const bool keep = (i < n) && ((int)strand[i] == want);
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m == 0) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (keep) {
            const unsigned long long o = base + __popc(m & ((1u << lane) - 1u));
            xs[o] = g_start[i];
            if (ye) ye[o] = g_end1[i];
        }
    }
}

__global__ void __launch_bounds__(TPB) iota_kernel(int64_t n, uint32_t* __restrict__ v) {
    const int64_t stride = (int64_t)gridDim.x * TPB;
    for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += stride)
        v[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(TPB)
gather_pairs_kernel(int64_t n, const uint32_t* __restrict__ perm,
                    const uint32_t* __restrict__ g_end1, const int8_t* __restrict__ strand,
                    uint32_t* __restrict__ p_end1, int8_t* __restrict__ p_strand) {
    const int64_t stride = (int64_t)gridDim.x * TPB;
    for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += stride) {
        const uint32_t j = perm[i];
        p_end1[i] = g_end1[j];
        if (p_strand) p_strand[i] = strand[j];
    }
}

// ---- running maximum over uint32 (three-kernel scan, tiles of 2048) ----------------------
constexpr int MX_ITEMS = 8;
constexpr int MX_TILE = TPB * MX_ITEMS;

__device__ __forceinline__ uint32_t block_max_scan(uint32_t v, uint32_t* total) {
    // inclusive running max over the block's threads
    __shared__ uint32_t wmax[TPB / 32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v = max(v, o);
    }
    if (lane == 31) wmax[warp] = v;
    __syncthreads();
    uint32_t pre = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < TPB / 32; w++) {
        uint32_t s = wmax[w];
        if (w < (int)warp) pre = max(pre, s);
        tot = max(tot, s);
    }
    __syncthreads();
    *total = tot;
    return max(pre, v);
}

__global__ void __launch_bounds__(TPB)
max_reduce_kernel(const uint32_t* __restrict__ in, int64_t n, uint32_t* __restrict__ partial) {
    const int64_t base = (int64_t)blockIdx.x * MX_TILE;
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < MX_ITEMS; k++) {
        int64_t i = base + (int64_t)k * TPB + threadIdx.x;
        if (i < n) m = max(m, in[i]);
    }
    uint32_t tot;
    block_max_scan(m, &tot);
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

// partial[b] <- max of all tiles BEFORE b (exclusive), one block
__global__ void __launch_bounds__(TPB)
max_partials_kernel(uint32_t* __restrict__ partial, int64_t nb) {
    uint32_t carry = 0;
    for (int64_t b0 = 0; b0 < nb; b0 += TPB) {
        int64_t i = b0 + threadIdx.x;
        uint32_t v = (i < nb) ? partial[i] : 0;
        uint32_t tot;
        uint32_t inc = block_max_scan(v, &tot);
        // exclusive = max over previous threads: recompute from the neighbour
        uint32_t prev = __shfl_up_sync(0xffffffffu, inc, 1);
        __shared__ uint32_t last_of_warp[TPB / 32];
        if ((threadIdx.x & 31) == 31) last_of_warp[threadIdx.x >> 5] = inc;
        __syncthreads();
        uint32_t ex;
        if ((threadIdx.x & 31) != 0) ex = prev;
        else ex = (threadIdx.x == 0) ? 0u : last_of_warp[(threadIdx.x >> 5) - 1];
        __syncthreads();
        if (i < nb) partial[i] = max(carry, ex);
        carry = max(carry, tot);
    }
}

__global__ void __launch_bounds__(TPB)
max_apply_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n,
                 const uint32_t* __restrict__ partial) {
    const int64_t base = (int64_t)blockIdx.x * MX_TILE + (int64_t)threadIdx.x * MX_ITEMS;
    uint32_t v[MX_ITEMS];
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < MX_ITEMS; k++) {
        int64_t i = base + k;
        v[k] = (i < n) ? in[i] : 0;
        m = max(m, v[k]);
    }
    uint32_t tot;
    uint32_t inc = block_max_scan(m, &tot);
    // running max of everything before this thread's first element
    uint32_t prev = __shfl_up_sync(0xffffffffu, inc, 1);
    __shared__ uint32_t last_of_warp[TPB / 32];
    if ((threadIdx.x & 31) == 31) last_of_warp[threadIdx.x >> 5] = inc;
    __syncthreads();
    uint32_t run;
    if ((threadIdx.x & 31) != 0) run = prev;
    else run = (threadIdx.x == 0) ? 0u : last_of_warp[(threadIdx.x >> 5) - 1];
    run = max(run, partial[blockIdx.x]);
#pragma unroll
    for (int k = 0; k < MX_ITEMS; k++) {
        int64_t i = base + k;
        run = max(run, v[k]);
        if (i < n) out[i] = run;
    }
}

int running_max_u32(const uint32_t* in, uint32_t* out, int64_t n) {
    if (n <= 0) return RCP_OK;
    const int64_t nb = (n + MX_TILE - 1) / MX_TILE;
    uint32_t* partial = nullptr;
    RCP_TRY(dalloc(&partial, (size_t)nb));
    max_reduce_kernel<<<(unsigned)nb, TPB, 0, g_ctx.stream>>>(in, n, partial);
    RCP_LAUNCHED();
    max_partials_kernel<<<1, TPB, 0, g_ctx.stream>>>(partial, nb);
    RCP_LAUNCHED();
    max_apply_kernel<<<(unsigned)nb, TPB, 0, g_ctx.stream>>>(in, out, n, partial);
    RCP_LAUNCHED();
    dfree(partial);
    return RCP_OK;
}

inline unsigned grid_for(int64_t n) {
    int64_t b = (n + TPB - 1) / TPB;
    int64_t cap = (int64_t)g_ctx.sm_count * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

}  // namespace

int running_max_u32_device(const uint32_t* in, uint32_t* out, int64_t n) { return running_max_u32(in, out, n); }

void reads_release(ReadsIdx& r) {
    if (r.bn_base) device_free(r.bn_base);
    r.bn_base = nullptr;
    r.bn_cand = r.bn_boff = r.bn_cb = nullptr;
    dfree(r.ln_xs);
    dfree(r.ln_e1);
    dfree(r.ln_st);
    dfree(r.ln_maxe1);
    r.ln_n = 0;
    dfree(r.pd_err);
    dfree(r.pd_cnt);
    dfree(r.pd_w);
    dfree(r.pd_run_first);
    r.pending = false;
    dfree(r.d_chrom_len);
    dfree(r.d_chrom_off);
    dfree(r.d_len_na);
    dfree(r.g_start);
    dfree(r.g_end1);
    dfree(r.d_strand);
    for (int c = 0; c < CLS_N; c++) {
        dfree(r.cls[c].xs);
        dfree(r.cls[c].ye);
        dfree(r.cls[c].cxs);
        dfree(r.cls[c].cye);
        r.cls[c].built = false;
        r.cls[c].xs_sorted = false;
    }
    dfree(r.exc_xw);
    dfree(r.exc_e1);
    dfree(r.exc_st);
    dfree(r.p_end1);
    dfree(r.p_strand);
    dfree(r.p_maxend1);
    r.pairs_built = false;
}

int reads_build_class(ReadsIdx& r, int cls) {
    SortedClass& sc = r.cls[cls];
    if (sc.built) return RCP_OK;
    const bool uni = r.uniform_w != 0;   // ye == xs + w: no second array, no second sort
    const bool xs_done = sc.xs_sorted;   // the pair sort of the GRangesList path already made xs
    if (cls == CLS_ALL) {
        sc.n = r.n;
        if (sc.xs == nullptr) {    // pre-filled by the map kernel under RCP_PATH_INDEX
            RCP_TRY(dalloc(&sc.xs, (size_t)r.n));
            RCP_CUDA(cudaMemcpyAsync(sc.xs, r.g_start, (size_t)r.n * 4, cudaMemcpyDeviceToDevice,
                                     g_ctx.stream));
        }
        if (!uni) {
            RCP_TRY(dalloc(&sc.ye, (size_t)r.n));
            RCP_CUDA(cudaMemcpyAsync(sc.ye, r.g_end1, (size_t)r.n * 4, cudaMemcpyDeviceToDevice,
                                     g_ctx.stream));
        }
    } else {
        // sc.n was filled from the strand histogram at load time
        RCP_TRY(dalloc(&sc.xs, (size_t)sc.n));
        if (!uni) RCP_TRY(dalloc(&sc.ye, (size_t)sc.n));
        if (sc.n > 0) {
            if (!r.has_strand) {   // every read is '*': the STAR class is everything
                RCP_CUDA(cudaMemcpyAsync(sc.xs, r.g_start, (size_t)r.n * 4,
                                         cudaMemcpyDeviceToDevice, g_ctx.stream));
                if (!uni)
                    RCP_CUDA(cudaMemcpyAsync(sc.ye, r.g_end1, (size_t)r.n * 4,
                                             cudaMemcpyDeviceToDevice, g_ctx.stream));
            } else {
                unsigned long long* cursor = nullptr;
                RCP_TRY(dalloc(&cursor, 1));
                RCP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long), g_ctx.stream));
                const int want = cls == CLS_PLUS ? 1 : (cls == CLS_MINUS ? -1 : 0);
                compact_strand_kernel<<<grid_for(r.n), TPB, 0, g_ctx.stream>>>(
                    r.n, r.g_start, r.g_end1, r.d_strand, want, sc.xs, sc.ye, cursor);
                RCP_LAUNCHED();
                dfree(cursor);
            }
        }
    }
    if (uni && r.n_exc > 0) {
        // reads whose width is not w: the main source assumed "end + 1 = start + w" for them;
        // the correction source cancels that event (+1 at start + w) and adds the true one
        sc.cn = r.n_exc;
        RCP_TRY(dalloc(&sc.cxs, (size_t)sc.cn));
        RCP_TRY(dalloc(&sc.cye, (size_t)sc.cn));
        const int want = cls == CLS_ALL ? 2 : (cls == CLS_PLUS ? 1 : (cls == CLS_MINUS ? -1 : 0));
        exc_select_kernel<<<(unsigned)((sc.cn + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(
            (uint32_t)sc.cn, r.exc_xw, r.exc_e1, r.exc_st, r.has_strand ? want : 2, sc.cxs, sc.cye);
        RCP_LAUNCHED();
    }
    {
        StageTimer t(ST_INDEX_SORT);
        if (!xs_done) RCP_TRY(sort_keys_u32(sc.xs, sc.n, r.key_bits));
        sc.xs_sorted = true;
        if (!uni) RCP_TRY(sort_keys_u32(sc.ye, sc.n, r.key_bits));
        if (sc.cn > 0) {
            RCP_TRY(sort_keys_u32(sc.cxs, sc.cn, 32));
            RCP_TRY(sort_keys_u32(sc.cye, sc.cn, 32));
        }
    }
    r.device_bytes += (size_t)sc.n * (uni ? 4 : 8);
    sc.built = true;
    return RCP_OK;
}

int reads_build_pairs(ReadsIdx& r) {
    if (r.pairs_built) return RCP_OK;
    // One (start, read id) pair sort gives both the permutation and the sorted starts the list
    // kernels search (the xs of the ALL class); the independently sorted ends of that class are
    // only needed by the rank method and stay unbuilt until a GRanges mask asks for them.
    SortedClass& all = r.cls[CLS_ALL];
    uint32_t *keys = nullptr, *perm = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)r.n));
    RCP_TRY(dalloc(&perm, (size_t)r.n));
    RCP_CUDA(cudaMemcpyAsync(keys, r.g_start, (size_t)r.n * 4, cudaMemcpyDeviceToDevice,
                             g_ctx.stream));
    iota_kernel<<<grid_for(r.n), TPB, 0, g_ctx.stream>>>(r.n, perm);
    RCP_LAUNCHED();
    {
        StageTimer t(ST_INDEX_SORT);
        RCP_TRY(sort_pairs_u32(keys, perm, r.n, r.key_bits));
    }
    if (!all.xs_sorted) {           // hand the sorted keys to the ALL class
        dfree(all.xs);
        all.xs = keys;
        all.n = r.n;
        all.xs_sorted = true;
        keys = nullptr;
    }
    RCP_TRY(dalloc(&r.p_end1, (size_t)r.n));
    if (r.has_strand) RCP_TRY(dalloc(&r.p_strand, (size_t)r.n));
    gather_pairs_kernel<<<grid_for(r.n), TPB, 0, g_ctx.stream>>>(r.n, perm, r.g_end1, r.d_strand,
                                                                r.p_end1, r.p_strand);
    RCP_LAUNCHED();
    RCP_TRY(dalloc(&r.p_maxend1, (size_t)r.n));
    RCP_TRY(running_max_u32(r.p_end1, r.p_maxend1, r.n));
    if (keys) dfree(keys);
    dfree(perm);
    r.device_bytes += (size_t)r.n * (8 + (r.has_strand ? 1 : 0));
    r.pairs_built = true;
    return RCP_OK;
}

// seqnames given as runs (GRanges keeps them as an Rle): run r covers reads
// [run_first[r], run_first[r + 1]).  Every thread writes four consecutive reads: a binary search
// places the first one, the others walk forward.  Reads beyond the runs' total get -1 (flagged by
// the map kernel as a bad chromosome id).
__global__ void __launch_bounds__(TPB)
rle_expand_kernel(int64_t n, int64_t n_runs, const int32_t* __restrict__ run_value,
                  const uint32_t* __restrict__ run_first /* n_runs + 1 */,
                  int32_t* __restrict__ dense /* padded to a multiple of 4 */) {
    const int64_t stride = (int64_t)gridDim.x * TPB;
    const int64_t n_vec = (n + 3) >> 2;
    for (int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x; v < n_vec; v += stride) {
        const uint32_t i0 = (uint32_t)(v * 4);
        int64_t a = 0, b = n_runs;              // largest run with run_first <= i0
        while (b - a > 1) {
            const int64_t mid = (a + b) >> 1;
            if (__ldg(run_first + mid) <= i0) a = mid;
            else b = mid;
        }
        int64_t r = a;
        uint32_t next = __ldg(run_first + r + 1);
        int32_t val = __ldg(run_value + r);
        int32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            while (i0 + k >= next && r + 1 < n_runs) {
                r++;
                next = __ldg(run_first + r + 1);
                val = __ldg(run_value + r);
            }
            o[k] = (i0 + k < next) ? val : -1;
        }
        reinterpret_cast<int4*>(dense)[v] = make_int4(o[0], o[1], o[2], o[3]);
    }
}

__global__ void __launch_bounds__(TPB)
rle_check_kernel(int64_t n_runs, const int32_t* __restrict__ run_len, unsigned int* __restrict__ err) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i < n_runs && run_len[i] < 0) atomicOr(err, 8u);
}

// Builds the raw global-coordinate arrays (and, under RCP_PATH_INDEX, the ALL class at once; it
// is otherwise built by the first call that needs it).  Synchronises once to validate.
// chrom == nullptr: the chromosome ids come as n_runs runs (run_chrom, run_len).
int reads_load_impl(ReadsIdx& r, int64_t n, const int32_t* chrom, int64_t n_runs,
                    const int32_t* run_chrom, const int32_t* run_len, const int32_t* start,
                    const int32_t* end, const int8_t* strand, int n_chrom,
                    const int64_t* chrom_len, int frag_len, int mem, int fixed_width) {
    const bool dbg = getenv("RCP_DEBUG_TIMING") != nullptr;
    auto t_start = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!dbg) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[rcp_reads_load] %-28s %8.3f ms\n", what,
                std::chrono::duration<double, std::milli>(now - t_start).count());
        t_start = now;
    };
    r.n = n;
    r.n_chrom = n_chrom;
    r.has_strand = strand != nullptr;
    r.chrom_len.assign(chrom_len, chrom_len + n_chrom);
    r.chrom_off.resize((size_t)n_chrom + 1);
    r.len_na.assign((size_t)n_chrom, 0);
    r.any_na = false;
    for (int c = 0; c < n_chrom; c++)
        if (chrom_len[c] <= 0) {            // NA: a stand-in follows from the reads (below)
            r.len_na[(size_t)c] = 1;
            r.any_na = true;
        }
    // chromosome layout in the global coordinate; with NA lengths it waits for the stand-ins
    auto layout = [&]() -> int {
        uint64_t off = 0;
        for (int c = 0; c < n_chrom; c++) {
            r.chrom_off[c] = (uint32_t)off;
            off += (uint64_t)r.chrom_len[(size_t)c] + 2;
            if (off >= 0xfffffff0ull)
                return fail(RCP_ERR_UNSUPPORTED,
                            "genome longer than 2^32 positions: 64-bit coordinates not implemented");
        }
        r.chrom_off[n_chrom] = (uint32_t)off;
        r.key_bits = 1;
        while (r.key_bits < 32 && (1ull << r.key_bits) <= off) r.key_bits++;
        RCP_CUDA(cudaMemcpyAsync(r.d_chrom_len, r.chrom_len.data(), (size_t)n_chrom * 8,
                                 cudaMemcpyHostToDevice, g_ctx.stream));
        RCP_CUDA(cudaMemcpyAsync(r.d_chrom_off, r.chrom_off.data(), ((size_t)n_chrom + 1) * 4,
                                 cudaMemcpyHostToDevice, g_ctx.stream));
        return RCP_OK;
    };
    RCP_TRY(dalloc(&r.d_chrom_len, (size_t)n_chrom));
    RCP_TRY(dalloc(&r.d_chrom_off, (size_t)n_chrom + 1));
    if (!r.any_na) RCP_TRY(layout());

    DevIn<int32_t> d_chrom, d_start, d_end, d_run_chrom, d_run_len;
    DevIn<int8_t> d_strand;
    const bool rle = chrom == nullptr && n > 0;
    if (rle) {
        RCP_TRY(d_run_chrom.init(run_chrom, (size_t)n_runs, mem));
        RCP_TRY(d_run_len.init(run_len, (size_t)n_runs, mem));
    } else {
        RCP_TRY(d_chrom.init(chrom, (size_t)n, mem));
    }
    RCP_TRY(d_start.init(start, (size_t)n, mem));
    RCP_TRY(d_end.init(end, (size_t)n, mem));            // nullptr with fixed_width: nothing to copy
    RCP_TRY(d_strand.init(strand, (size_t)n, mem));
    lap("staging copies enqueued");

    RCP_TRY(dalloc(&r.g_start, (size_t)n));
    RCP_TRY(dalloc(&r.g_end1, (size_t)n));
    if (r.has_strand) RCP_TRY(dalloc(&r.d_strand, (size_t)n));
    unsigned int* d_err = nullptr;
    unsigned long long* d_cnt = nullptr;
    unsigned int* d_w = nullptr;    // [0] exception count, [1] candidate width, [2] reads wider than long_thr
    RCP_TRY(dalloc(&d_err, 1));
    RCP_TRY(dalloc(&d_cnt, 4));
    RCP_TRY(dalloc(&d_w, 4));
    RCP_CUDA(cudaMemsetAsync(d_err, 0, sizeof(unsigned int), g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(d_cnt, 0, 4 * sizeof(unsigned long long), g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(d_w, 0, 4 * sizeof(unsigned int), g_ctx.stream));
    uint32_t* run_first = nullptr;      // exclusive scan of the run lengths + their total
    if (rle) {
        StageTimer t(ST_INDEX_MAP);
        RCP_TRY(dalloc(&run_first, (size_t)n_runs + 1));
        RCP_TRY(dalloc(&d_chrom.owned, ((size_t)n + 3) & ~(size_t)3));
        d_chrom.ptr = d_chrom.owned;
        rle_check_kernel<<<(unsigned)((n_runs + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(n_runs, d_run_len.ptr, d_err);
        RCP_LAUNCHED();
        RCP_TRY(exclusive_scan_u32(reinterpret_cast<const uint32_t*>(d_run_len.ptr), run_first, n_runs,
                                   run_first + n_runs));
        rle_expand_kernel<<<grid_for((n + 3) / 4), TPB, 0, g_ctx.stream>>>(
            n, n_runs, d_run_chrom.ptr, run_first, d_chrom.owned);
        RCP_LAUNCHED();
    }
    if (r.any_na) {
        // stand-in lengths: the largest (extended) read end of each NA chromosome -- one pass over
        // the reads and one host synchronisation that samples with known seqlengths never pay
        unsigned long long* d_max = nullptr;
        RCP_TRY(dalloc(&d_max, (size_t)n_chrom));
        RCP_CUDA(cudaMemsetAsync(d_max, 0, (size_t)n_chrom * 8, g_ctx.stream));
        if (n > 0) {
            chrom_max_end_kernel<<<grid_for(n), TPB, 0, g_ctx.stream>>>(n, d_chrom.ptr, d_start.ptr, d_end.ptr,
                                                                       d_strand.ptr, n_chrom, frag_len, fixed_width,
                                                                       d_max);
            RCP_LAUNCHED();
        }
        std::vector<unsigned long long> h_max((size_t)n_chrom, 0ull);
        RCP_CUDA(cudaMemcpyAsync(h_max.data(), d_max, (size_t)n_chrom * 8, cudaMemcpyDeviceToHost, g_ctx.stream));
        RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        dfree(d_max);
        for (int c = 0; c < n_chrom; c++)
            if (r.len_na[(size_t)c])
                r.chrom_len[(size_t)c] = (int64_t)std::min<unsigned long long>(std::max<unsigned long long>(h_max[(size_t)c], 1ull),
                                                                               0x7ffffff0ull);
        RCP_TRY(layout());
        RCP_TRY(dalloc(&r.d_len_na, (size_t)n_chrom));
        RCP_CUDA(cudaMemcpyAsync(r.d_len_na, r.len_na.data(), (size_t)n_chrom, cudaMemcpyHostToDevice, g_ctx.stream));
    }
    {   // the widest read the split path's packed word holds for this genome (coverage_split.cu)
        const int wbits = 32 - split_position_bits((int64_t)r.chrom_off[(size_t)n_chrom]) - (r.has_strand ? 2 : 0);
        r.long_thr = wbits >= 7 ? std::min<uint32_t>((1u << wbits) - 1u, 8191u) : 0xffffffffu;
    }
    ExcBuf exc;
    // (the exception counter is ONE address: a sample whose widths vary hits it once per read
    // until the buffer is full, so the buffer stays small)
    exc.cap = (uint32_t)std::min<int64_t>(std::max<int64_t>(n / 64, 4096), 65536);
    RCP_TRY(dalloc(&r.exc_xw, (size_t)exc.cap));
    RCP_TRY(dalloc(&r.exc_e1, (size_t)exc.cap));
    RCP_TRY(dalloc(&r.exc_st, (size_t)exc.cap));
    exc.xw = r.exc_xw;
    exc.e1 = r.exc_e1;
    exc.st = r.exc_st;
    exc.count = d_w;
    exc.w_out = d_w + 1;
    // RCP_PATH_INDEX: the map kernel also writes the copy of g_start the index sort works on
    const bool eager_index = g_ctx.coverage_path == RCP_PATH_INDEX;
    if (eager_index) RCP_TRY(dalloc(&r.cls[CLS_ALL].xs, (size_t)n));
    if (n > 0) {
        StageTimer t(ST_INDEX_MAP);
        auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
        const bool vec = al16(d_chrom.ptr) && al16(d_start.ptr) && (d_end.ptr == nullptr || al16(d_end.ptr)) &&
                         (d_strand.ptr == nullptr || (reinterpret_cast<uintptr_t>(d_strand.ptr) & 3u) == 0);
        const unsigned grid = grid_for(vec ? (n + 3) / 4 : n);
        auto launch = [&](auto kern) {
            kern<<<grid, TPB, 0, g_ctx.stream>>>(n, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr, r.d_chrom_off,
                                                 r.d_chrom_len, n_chrom, frag_len, fixed_width, r.long_thr, r.g_start,
                                                 r.g_end1,
                                                 r.cls[CLS_ALL].xs, r.d_strand, d_err, d_cnt, exc);
        };
        if (d_end.ptr) {
            if (vec) launch(reads_to_global_kernel<4, true>);
            else launch(reads_to_global_kernel<1, true>);
        } else {
            if (vec) launch(reads_to_global_kernel<4, false>);
            else launch(reads_to_global_kernel<1, false>);
        }
        RCP_LAUNCHED();
    }
    lap("map kernel enqueued");
    r.pending = true;
    r.pd_rle = rle;
    r.pd_err = d_err;
    r.pd_cnt = d_cnt;
    r.pd_w = d_w;
    r.pd_run_first = run_first;
    r.pd_run_total = rle ? run_first + n_runs : nullptr;
    r.pd_exc_cap = exc.cap;
    r.pd_eager_index = eager_index;
    r.device_bytes += (size_t)n * (8 + (r.has_strand ? 1 : 0));
    // Deferred validation: the status words stay on the device until the first call that uses
    // the handle reads them (that call reports a data error of these reads).
    if (g_ctx.deferred_validation && !eager_index) return RCP_OK;
    RCP_TRY(reads_resolve(r));
    lap("sync (copies + map kernel)");
    return RCP_OK;
}

int reads_pending_items(ReadsIdx& r, FetchItem* items, int* n) {
    if (!r.pending) return RCP_OK;
    items[(*n)++] = {r.pd_err, &r.h_err, 4};
    items[(*n)++] = {r.pd_cnt, r.h_cnt, 32};
    items[(*n)++] = {r.pd_w, r.h_w, 16};
    if (r.pd_rle) items[(*n)++] = {r.pd_run_total, &r.h_total, 4};
    return RCP_OK;
}

int reads_resolve(ReadsIdx& r) {
    if (r.pending) {
        FetchItem items[4];
        int n = 0;
        reads_pending_items(r, items, &n);
        RCP_TRY(fetch_and_sync(items, n));
    }
    return reads_finish(r);
}

namespace {

// what follows the fetch of the status words (the caller has synchronised)
int finish_pending(ReadsIdx& r) {
    const int64_t n = r.n;
    const unsigned int h_err = r.h_err;
    dfree(r.pd_err);
    dfree(r.pd_cnt);
    dfree(r.pd_w);
    dfree(r.pd_run_first);
    r.pd_run_total = nullptr;
    if (h_err & 8u) return fail(RCP_ERR_DATA, "a seqnames run has a negative length");
    if (r.pd_rle && (int64_t)r.h_total != n)
        return fail(RCP_ERR_DATA, "the seqnames run lengths sum to %u, not to the %lld reads", r.h_total,
                    (long long)n);
    // (nearly) every read has the same width w -- fixed-length or fragment-extended libraries;
    // the few that do not (trimmed at a chromosome end) live in a correction source.  Then the
    // sorted ends are the sorted starts shifted by w: one array, one sort.  (start + w must not
    // wrap around 2^32: a genome that ends within w of it keeps the second array.)
    const bool w_fits = (uint64_t)r.chrom_off[(size_t)r.n_chrom] + r.h_w[1] <= 0xffffffffull;
    if (h_err == 0 && n > 0 && r.h_w[1] > 0 && r.h_w[0] <= r.pd_exc_cap && w_fits) {
        r.uniform_w = r.h_w[1];
        r.n_exc = (int64_t)r.h_w[0];
    } else {
        r.uniform_w = 0;
        r.n_exc = 0;
    }
    if (r.n_exc == 0) {
        dfree(r.exc_xw);
        dfree(r.exc_e1);
        dfree(r.exc_st);
    }
    if (h_err & 1u) return fail(RCP_ERR_DATA, "a read has a chromosome id outside [0, n_chrom)");
    if (h_err & 2u) return fail(RCP_ERR_DATA, "a read violates 1 <= start <= end");
    if (h_err & 4u) return fail(RCP_ERR_DATA, "a read starts beyond the end of its chromosome");
    r.cls[CLS_PLUS].n = (int64_t)r.h_cnt[0];
    r.cls[CLS_MINUS].n = (int64_t)r.h_cnt[1];
    r.cls[CLS_STAR].n = (int64_t)r.h_cnt[2];
    r.max_width = (uint32_t)r.h_cnt[3];
    r.n_long = (int64_t)r.h_w[2];
    if (r.pd_eager_index) RCP_TRY(reads_build_class(r, CLS_ALL));
    return RCP_OK;
}

}  // namespace

// A failed validation leaves the handle without its widths and class counts, so its error is kept
// and returned again by every later call: a retry must not compute a coverage from such a handle.
int reads_finish(ReadsIdx& r) {
    if (r.pending) {
        r.pending = false;
        const int rc = finish_pending(r);
        if (rc != RCP_OK) {
            r.failed = rc;
            r.failed_msg = rcp_last_error();
        }
        return rc;
    }
    if (r.failed != RCP_OK) return fail(r.failed, "%s", r.failed_msg.c_str());
    return RCP_OK;
}

// ---- ranges[-which(width > qu)][idx] followed by the load (SURVEY 8f N3) ----------------------
namespace {

__global__ void __launch_bounds__(TPB)
keep_flags_kernel(int64_t n, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                  double max_width, uint32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;
    const double w = (double)end[i] - (double)start[i] + 1.0;
    flag[i] = !(w > max_width);
}

// kept_pos[rank of read i among the kept] = i
__global__ void __launch_bounds__(TPB)
kept_positions_kernel(int64_t n, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ rank,
                      uint32_t* __restrict__ kept_pos) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i < n && flag[i]) kept_pos[rank[i]] = (uint32_t)i;
}

// out[j] = in[ kept_pos[ idx[j] - 1 ] ]   (either level of indirection may be absent)
__global__ void __launch_bounds__(TPB)
select_gather_kernel(int64_t k, int64_t n_kept, const int32_t* __restrict__ idx,
                     const uint32_t* __restrict__ kept_pos, const int32_t* __restrict__ chrom,
                     const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                     const int8_t* __restrict__ strand, int32_t* __restrict__ o_chrom,
                     int32_t* __restrict__ o_start, int32_t* __restrict__ o_end,
                     int8_t* __restrict__ o_strand, unsigned int* __restrict__ err) {
    const int64_t j = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (j >= k) return;
    int64_t p = idx ? (int64_t)idx[j] - 1 : j;
    if (p < 0 || p >= n_kept) {
        atomicOr(err, 1u);
        p = 0;
    }
    const int64_t i = kept_pos ? (int64_t)kept_pos[p] : p;
    o_chrom[j] = chrom[i];
    o_start[j] = start[i];
    o_end[j] = end[i];
    if (o_strand) o_strand[j] = strand[i];
}

}  // namespace

int reads_load_select_impl(ReadsIdx& r, int64_t n, const int32_t* chrom, const int32_t* start,
                           const int32_t* end, const int8_t* strand, double max_width, int64_t k,
                           const int32_t* idx, int n_chrom, const int64_t* chrom_len, int frag_len,
                           int mem, int64_t* n_kept_out) {
    DevIn<int32_t> d_chrom, d_start, d_end, d_idx;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_chrom.init(chrom, (size_t)n, mem));
    RCP_TRY(d_start.init(start, (size_t)n, mem));
    RCP_TRY(d_end.init(end, (size_t)n, mem));
    RCP_TRY(d_strand.init(strand, (size_t)n, mem));
    RCP_TRY(d_idx.init(idx, (size_t)k, mem));
    const bool filter = max_width >= 0.0 && n > 0;
    int64_t n_kept = n;
    uint32_t *flag = nullptr, *rank = nullptr, *kept_pos = nullptr;
    unsigned int* d_err = nullptr;
    RCP_TRY(dalloc(&d_err, 1));
    RCP_CUDA(cudaMemsetAsync(d_err, 0, 4, g_ctx.stream));
    int rc = RCP_OK;
    if (filter) {
        StageTimer t(ST_INDEX_MAP);
        rc = dalloc(&flag, (size_t)n);
        if (rc == RCP_OK) rc = dalloc(&rank, (size_t)n + 1);
        if (rc == RCP_OK) {
            keep_flags_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(n, d_start.ptr, d_end.ptr, max_width, flag);
            g_ctx.launches++;
            rc = exclusive_scan_u32(flag, rank, n, rank + n);
        }
        uint32_t h_kept = 0;
        if (rc == RCP_OK) {
            cudaError_t e = cudaMemcpyAsync(&h_kept, rank + n, 4, cudaMemcpyDeviceToHost, g_ctx.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "width filter failed: %s", cudaGetErrorString(e));
        }
        n_kept = (int64_t)h_kept;
        if (rc == RCP_OK) rc = dalloc(&kept_pos, (size_t)n_kept);
        if (rc == RCP_OK && n_kept > 0) {
            kept_positions_kernel<<<(unsigned)((n + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(n, flag, rank, kept_pos);
            g_ctx.launches++;
        }
    }
    if (n_kept_out) *n_kept_out = n_kept;
    const int64_t m = idx ? k : n_kept;                 // reads that reach the load
    int32_t *o_chrom = nullptr, *o_start = nullptr, *o_end = nullptr;
    int8_t* o_strand = nullptr;
    if (rc == RCP_OK) rc = dalloc(&o_chrom, (size_t)m);
    if (rc == RCP_OK) rc = dalloc(&o_start, (size_t)m);
    if (rc == RCP_OK) rc = dalloc(&o_end, (size_t)m);
    if (rc == RCP_OK && strand) rc = dalloc(&o_strand, (size_t)m);
    unsigned int h_err = 0;
    if (rc == RCP_OK && m > 0) {
        if (n_kept == 0) {
            rc = fail(RCP_ERR_DATA, "an index selects from an empty set of reads");
        } else {
            StageTimer t(ST_INDEX_MAP);
            select_gather_kernel<<<(unsigned)((m + TPB - 1) / TPB), TPB, 0, g_ctx.stream>>>(
                m, n_kept, d_idx.ptr, kept_pos, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr, o_chrom,
                o_start, o_end, o_strand, d_err);
            g_ctx.launches++;
            cudaError_t e = cudaMemcpyAsync(&h_err, d_err, 4, cudaMemcpyDeviceToHost, g_ctx.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "read selection failed: %s", cudaGetErrorString(e));
            if (rc == RCP_OK && h_err)
                rc = fail(RCP_ERR_DATA, "a selection index is outside 1..%lld", (long long)n_kept);
        }
    }
    if (rc == RCP_OK)
        rc = reads_load_impl(r, m, o_chrom, 0, nullptr, nullptr, o_start, o_end, o_strand, n_chrom, chrom_len,
                             frag_len, RCP_MEM_DEVICE, 0);
    dfree(flag);
    dfree(rank);
    dfree(kept_pos);
    dfree(d_err);
    dfree(o_chrom);
    dfree(o_start);
    dfree(o_end);
    dfree(o_strand);
    return rc;
}

}  // namespace rcp
