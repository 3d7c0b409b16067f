// Coverage kernels (sm_100a): calcCoverage / coverageFromRanges of the reference
// (/root/reference/R/coverage.R:126-226) over the rank index built by index.cu.
//
// For a window [gs, ge] in global coordinates and sorted arrays xs (starts), ye (ends+1):
//     reads overlapping the window   n_ov = #{xs <= ge} - #{ye <= gs}          (NULL rule)
//     coverage entering a tile at t  base = #{xs <  t} - #{ye <  t}
//     inside the tile                diff[p-t] = #{xs == p} - #{ye == p},  cov = base + cumsum
// so a tile needs only two contiguous slices of xs and ye (found by binary search), a
// shared-memory difference array filled with warp-aggregated atomics, a block prefix scan and
// one coalesced int32 store (reversed for '-' regions, coverage.R:212-213).  Tiles of one
// region are independent: no carry is passed between CTAs.
//
//   region_plan_kernel   1 thread / region : geometry checks, NULL rule, slice bounds
//   cov_small_kernel     1 warp  / region  : regions of <= 1024 bp (warp-private smem tile)
//   cov_tile_kernel      1 CTA   / tile    : longer regions cut into <= 4096-bp tiles
//   list_plan_kernel / cov_list_kernel     : GRangesList elements (exons stitched per gene,
//                                            read multiplicity, coverage.R:202-207)
#include "cov_common.cuh"
#include "rcp_internal.cuh"

namespace rcp {

using namespace covk;

namespace {

// ye[i] is read as ye[i] + yshift: in uniform-width mode ye aliases xs and yshift is the width.
template <int NS>
struct Sources {
    const uint32_t* xs[NS];
    const uint32_t* ye[NS];
    uint32_t n[NS];
    uint32_t yshift[NS];
    uint8_t cls_bit[NS];   // bit of the region's class mask that enables this source
    uint8_t corr[NS];      // 1: correction source of the uniform-width index (index.cu)
};

struct RegionArrays {
    // outputs of the plan kernel, one entry per region (x NS where noted)
    uint32_t* gs;        // global coordinate of the first base
    int32_t* len;        // 0 for NULL
    uint8_t* flags;      // bit0 reverse, bits1..3 class mask
    uint8_t* is_null;
    uint32_t* ix0;       // [R*NS] lower_bound(xs, gs)
    uint32_t* ix1;       // [R*NS] lower_bound(xs, ge+1)
    uint32_t* iy0;       // [R*NS] lower_bound(ye, gs)
    uint32_t* iy1;       // [R*NS] lower_bound(ye, ge+1)
    int64_t* padded;     // padded length (scan input)
    int64_t* ntiles;     // tiles of the CTA kernel (scan input)
};

// first index in [lo, hi) with a[idx] + shift >= key
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* __restrict__ a, uint32_t lo,
                                                    uint32_t hi, uint32_t key, uint32_t shift = 0) {
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) + shift < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// The same search done by a whole warp, 32 probes per step (all lanes pass the same arguments
// and receive the same answer): a slice of a few thousand reads resolves in 2-3 dependent loads
// instead of ~12.
__device__ __forceinline__ uint32_t warp_lower_bound_u32(const uint32_t* __restrict__ a,
                                                         uint32_t lo, uint32_t hi, uint32_t key,
                                                         uint32_t shift) {
    const uint32_t lane = threadIdx.x & 31;
    while (lo < hi) {
        const uint32_t step = (hi - lo + 31u) >> 5;
        const uint32_t p = lo + (lane + 1u) * step - 1u;       // last element of chunk `lane`
        const bool ge = (p < hi) ? (__ldg(a + p) + shift >= key) : true;
        const unsigned b = __ballot_sync(0xffffffffu, ge);     // chunks past hi vote true
        if (b == 0u) return hi;                                // all 32 chunks in range and < key
        const uint32_t f = (uint32_t)__ffs(b) - 1u;
        const uint32_t pf = lo + (f + 1u) * step - 1u;
        lo += f * step;
        if (pf < hi) hi = pf;          // a[pf] >= key: answer in [lo, pf]
        else if (lo >= hi) return hi;  // every probed chunk was < key and nothing is left
        // else: the unprobed tail chunk [lo, hi) remains (shorter than step)
    }
    return lo;
}

// lower_bound started from a nearby position `hint` (exponential probe, then bisection): the
// five ranks a region needs lie within a few hundred reads of each other.
__device__ __forceinline__ uint32_t gallop_lower_bound_u32(const uint32_t* __restrict__ a,
                                                           uint32_t n, uint32_t hint,
                                                           uint32_t key, uint32_t shift) {
    if (n == 0) return 0;
    if (hint >= n) hint = n - 1;
    uint32_t lo, hi;
    if (__ldg(a + hint) + shift < key) {          // answer in (hint, n]
        lo = hint + 1;
        uint32_t step = 1;
        while (lo + step <= n && __ldg(a + lo + step - 1) + shift < key) {
            lo += step;
            step <<= 1;
        }
        hi = min(lo + step, n);
        // invariant: everything before lo is < key; a[hi-1] >= key or hi == n
    } else {                                      // answer in [0, hint]
        hi = hint;
        uint32_t step = 1;
        while (hi >= step && __ldg(a + hi - step) + shift >= key) {
            hi -= step;
            step <<= 1;
        }
        lo = hi >= step ? hi - step + 1 : 0;
    }
    return lower_bound_u32(a, lo, hi, key, shift);
}

// err bits: 1 chrom id out of range, 2 end < start - 1
// One thread per region.  Only the first rank is a full-range bisection; the other four gallop
// from it.
template <int NS>
__global__ void __launch_bounds__(CTA)
region_plan_kernel(int64_t R, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
                   const int32_t* __restrict__ end, const int8_t* __restrict__ strand,
                   const uint32_t* __restrict__ chrom_off, const int64_t* __restrict__ chrom_len,
                   int n_chrom, Sources<NS> src, int ignore_strand, int strand_filter,
                   RegionArrays out, unsigned int* __restrict__ err,
                   unsigned long long* __restrict__ stats /* [0] n_null, [1] total_len */) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (r < R) {
        const int c = chrom[r];
        const int64_t s = start[r], e = end[r];
        const int st = strand ? (int)strand[r] : 0;
        uint32_t gs = 0;
        int64_t L = 0;
        const unsigned mask = NS <= 2 ? 1u : class_mask(st, ignore_strand, strand_filter);
        bool null = window_geometry(c, s, e, n_chrom, chrom_off, chrom_len, err, &gs, &L);
        if (!null) {
            const uint32_t ge = gs + (uint32_t)(L - 1);
            long long nov = 0;
#pragma unroll
            for (int k = 0; k < NS; k++) {
                uint32_t x0 = 0, x1 = 0, y0 = 0, y1 = 0;
                if ((mask >> src.cls_bit[k]) & 1u) {
                    const uint32_t n = src.n[k];
                    const uint32_t sh = src.yshift[k];
                    x0 = lower_bound_u32(src.xs[k], 0, n, gs);
                    x1 = gallop_lower_bound_u32(src.xs[k], n, x0, ge + 1u, 0);
                    y0 = gallop_lower_bound_u32(src.ye[k], n, x0, gs, sh);
                    const uint32_t yov = gallop_lower_bound_u32(src.ye[k], n, y0, gs + 1u, sh);
                    y1 = gallop_lower_bound_u32(src.ye[k], n, x1, ge + 1u, sh);
                    // reads overlapping the window: #{start <= ge} - #{end < gs}.  A correction
                    // source only moves end events, so both of its counts are taken at gs.
                    const uint32_t xov = src.corr[k] ? lower_bound_u32(src.xs[k], x0, x1, gs + 1u) : x1;
                    nov += (long long)xov - (long long)yov;
                }
                out.ix0[r * NS + k] = x0;
                out.ix1[r * NS + k] = x1;
                out.iy0[r * NS + k] = y0;
                out.iy1[r * NS + k] = y1;
            }
            if (nov <= 0) null = true;          // coverage.R:198,224-225
        }
        const int32_t len = null ? 0 : (int32_t)L;
        out.gs[r] = gs;
        out.len[r] = len;
        out.flags[r] = (uint8_t)((st < 0 ? 1u : 0u) | (mask << 1));
        out.is_null[r] = null ? 1 : 0;
        out.padded[r] = ((int64_t)len + PAD - 1) / PAD * PAD;
        out.ntiles[r] = len > SMALL_MAX ? ((int64_t)len + TILE - 1) / TILE : 0;
        my_null = null ? 1 : 0;
        my_len = (unsigned long long)len;
    }
    unsigned long long my_max = my_len;
    for (int d = 16; d > 0; d >>= 1) {
        my_null += __shfl_xor_sync(0xffffffffu, my_null, d);
        my_len += __shfl_xor_sync(0xffffffffu, my_len, d);
        my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
    }
    if ((threadIdx.x & 31) == 0) {
        if (my_null) atomicAdd(&stats[0], my_null);
        if (my_len) atomicAdd(&stats[1], my_len);
        if (my_max) atomicMax(&stats[2], my_max);
    }
}

__global__ void __launch_bounds__(CTA)
fill_tiles_kernel(int64_t R, const int64_t* __restrict__ ntiles,
                  const int64_t* __restrict__ tile_off, int32_t* __restrict__ tile_region) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= R) return;
    const int64_t n = ntiles[r], o = tile_off[r];
    for (int64_t j = 0; j < n; j++) tile_region[o + j] = (int32_t)r;
}

// ---- shared device pieces -------------------------------------------------------------------

// Add `sign` once per valid lane to diff[pos]; lanes hold NON-DECREASING positions (they walk a
// sorted array), so equal positions sit in adjacent lanes and one atomic per run is enough.
__device__ __forceinline__ void warp_aggregated_add(int* diff, uint32_t pos, bool valid,
                                                    int sign) {
    const unsigned lane = threadIdx.x & 31;
    const uint32_t key = valid ? pos : 0xffffffffu;
    const uint32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = (lane == 0) || (key != prev);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (head && valid) {
        const unsigned above = heads & ~((2u << lane) - 1u);
        const int run_end = above ? (__ffs(above) - 1) : 32;
        atomicAdd(diff + pos, sign * (run_end - (int)lane));
    }
}

// ---- warp-per-region kernel (L <= SMALL_MAX) -----------------------------------------------
template <int NS>
__global__ void __launch_bounds__(CTA)
cov_small_kernel(int64_t R, RegionArrays ra, Sources<NS> src, const int64_t* __restrict__ off,
                 int32_t* __restrict__ cov) {
    __shared__ __align__(16) int sm[WARPS][SMALL_MAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * WARPS + warp;
    if (r >= R) return;
    const int L = ra.len[r];
    if (L == 0 || L > SMALL_MAX) return;
    int* diff = sm[warp];
    const int nrows = (L + ROW - 1) / ROW;
    for (int i = lane; i < nrows * (ROW / 4); i += 32)
        reinterpret_cast<int4*>(diff)[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    const uint32_t gs = ra.gs[r];
    const unsigned flags = ra.flags[r];
    const unsigned mask = flags >> 1;
    const bool rev = (flags & 1u) != 0;
    const uint32_t last = (uint32_t)(L - 1);
    int base = 0, total = 0;
#pragma unroll
    for (int k = 0; k < NS; k++) {
        if (!((mask >> src.cls_bit[k]) & 1u)) continue;
        const uint32_t x0 = ra.ix0[r * NS + k], x1 = ra.ix1[r * NS + k];
        const uint32_t y0 = ra.iy0[r * NS + k], y1 = ra.iy1[r * NS + k];
        base += (int)(x0 - y0);
        total += (int)(x1 - x0) - (int)(y1 - y0);
        for (uint32_t i0 = x0; i0 < x1; i0 += 32) {
            const uint32_t i = i0 + lane;
            const bool ok = i < x1;
            uint32_t p = ok ? (__ldg(src.xs[k] + i) - gs) : 0u;
            if (rev) p = last - p;
            warp_aggregated_add(diff, p, ok, +1);
        }
        for (uint32_t i0 = y0; i0 < y1; i0 += 32) {
            const uint32_t i = i0 + lane;
            const bool ok = i < y1;
            uint32_t p = ok ? (__ldg(src.ye[k] + i) + src.yshift[k] - gs) : 0u;
            if (rev) p = last - p;
            warp_aggregated_add(diff, p, ok, -1);
        }
    }
    __syncwarp();
    int32_t* dst = cov + off[r];
    const int top = rev ? base + total : base;
    int pre = 0;
    for (int row = 0; row < nrows; row++)
        pre += warp_row_scan_store(diff + row * ROW, pre, top, rev, L - row * ROW, dst + row * ROW);
}

// ---- CTA-per-tile kernel --------------------------------------------------------------------
// Tiles are cut in OUTPUT space (tile j = outputs [j*tile_len, ...)), so a '-' region's tile j
// covers the genomic positions [L - o_hi, L - o_lo).
template <int NS>
__global__ void __launch_bounds__(CTA)
cov_tile_kernel(const int32_t* __restrict__ tile_region, const int64_t* __restrict__ tile_off,
                RegionArrays ra, Sources<NS> src, const int64_t* __restrict__ off,
                int32_t* __restrict__ cov) {
    __shared__ __align__(16) int diff[TILE];
    __shared__ int rowpre[MAX_ROWS + 1];
    __shared__ uint32_t bnd[4 * NS];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r = tile_region[blockIdx.x];
    const int j = (int)((int64_t)blockIdx.x - tile_off[r]);
    const int L = ra.len[r];
    const int m = (L + TILE - 1) / TILE;
    const int tile_len = (((L + m - 1) / m) + ROW - 1) / ROW * ROW;
    const int o_lo = j * tile_len;
    const int tlen = min(tile_len, L - o_lo);
    const unsigned flags = ra.flags[r];
    const unsigned mask = flags >> 1;
    const bool rev = (flags & 1u) != 0;
    const int q0 = rev ? (L - o_lo - tlen) : o_lo;          // genomic offset of the tile
    const uint32_t gts = ra.gs[r] + (uint32_t)q0;
    const uint32_t last = (uint32_t)(tlen - 1);
    // slice bounds of this tile, searched warp-wide inside the region's own slices
    for (int q = warp; q < 4 * NS; q += WARPS) {
        const int k = q >> 2, which = q & 3;
        const bool is_x = which < 2;
        const uint32_t key = (which & 1) ? gts + (uint32_t)tlen : gts;
        const uint32_t lo = is_x ? ra.ix0[r * NS + k] : ra.iy0[r * NS + k];
        const uint32_t hi = is_x ? ra.ix1[r * NS + k] : ra.iy1[r * NS + k];
        uint32_t res = lo;
        if ((mask >> src.cls_bit[k]) & 1u) {
            if (m == 1) res = (which & 1) ? hi : lo;
            else res = warp_lower_bound_u32(is_x ? src.xs[k] : src.ye[k], lo, hi, key,
                                            is_x ? 0u : src.yshift[k]);
        }
        if (lane == 0) bnd[q] = res;
    }
    const int nrows = (tlen + ROW - 1) / ROW;
    for (int i = tid; i < nrows * (ROW / 4); i += CTA)
        reinterpret_cast<int4*>(diff)[i] = make_int4(0, 0, 0, 0);
    __syncthreads();
    int base = 0;
#pragma unroll
    for (int k = 0; k < NS; k++) {
        if (!((mask >> src.cls_bit[k]) & 1u)) continue;
        const uint32_t x0 = bnd[4 * k + 0], x1 = bnd[4 * k + 1];
        const uint32_t y0 = bnd[4 * k + 2], y1 = bnd[4 * k + 3];
        base += (int)(x0 - y0);
        for (uint32_t i0 = x0 + warp * 32; i0 < x1; i0 += CTA) {
            const uint32_t i = i0 + lane;
            const bool ok = i < x1;
            uint32_t p = ok ? (__ldg(src.xs[k] + i) - gts) : 0u;
            if (rev) p = last - p;
            warp_aggregated_add(diff, p, ok, +1);
        }
        for (uint32_t i0 = y0 + warp * 32; i0 < y1; i0 += CTA) {
            const uint32_t i = i0 + lane;
            const bool ok = i < y1;
            uint32_t p = ok ? (__ldg(src.ye[k] + i) + src.yshift[k] - gts) : 0u;
            if (rev) p = last - p;
            warp_aggregated_add(diff, p, ok, -1);
        }
    }
    __syncthreads();
    block_scan_store(diff, tlen, base, rev, rowpre, cov + off[r] + o_lo);
}

// ---- GRangesList elements -------------------------------------------------------------------
struct ListArrays {
    // per range (exon), global coordinates
    uint32_t* xgs;       // global start (after the zero-index drop)
    uint32_t* xge;       // global end; xge < xgs marks a zero-width range
    int32_t* xoff;       // offset of the range inside the stitched element
    // per element
    int32_t* len;
    uint8_t* flags;      // bit0 reverse
    uint8_t* is_null;
    uint32_t* clo;       // candidate reads [clo, chi) in start-sorted order
    uint32_t* chi;
    uint32_t* span_lo;   // global start of the leftmost range
    int64_t* padded;
    int64_t* ntiles;
};

// err bits: 1 chrom id, 2 end < start-1, 4 ranges of one element on different chromosomes
__global__ void __launch_bounds__(CTA)
list_plan_kernel(int64_t G, const int64_t* __restrict__ ptr, const int32_t* __restrict__ chrom,
                 const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                 const int8_t* __restrict__ strand, const uint32_t* __restrict__ chrom_off,
                 const int64_t* __restrict__ chrom_len, int n_chrom,
                 const uint32_t* __restrict__ xs, const uint32_t* __restrict__ p_end1,
                 const int8_t* __restrict__ p_strand, const uint32_t* __restrict__ p_maxend1,
                 uint32_t n_reads, int ignore_strand, int strand_filter, ListArrays out,
                 unsigned int* __restrict__ err, unsigned long long* __restrict__ stats) {
    const int64_t g = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (g < G) {
        const int64_t a = ptr[g], b = ptr[g + 1];
        bool null = (b <= a);
        int64_t L = 0;
        uint32_t lo = 0xffffffffu, hi = 0;
        int st0 = 0;
        if (!null) {
            const int c = chrom[a];
            st0 = strand ? (int)strand[a] : 0;
            if (c < 0 || c >= n_chrom) {
                atomicOr(err, 1u);
                null = true;
            } else {
                const int64_t clen = chrom_len[c];
                const uint32_t coff = chrom_off[c];
                for (int64_t i = a; i < b; i++) {
                    int64_t s = start[i], e = end[i];
                    if (chrom[i] != c) atomicOr(err, 4u);
                    if (e < s - 1) { atomicOr(err, 2u); null = true; }
                    if (s < 0 || e > clen) null = true;      // coverage.R:206 inside tryCatch
                    if (s == 0) s = 1;
                    int64_t w = e - s + 1;
                    if (w < 0) w = 0;
                    const uint32_t gs = coff + (uint32_t)(s > 0 ? s : 0);
                    out.xgs[i] = gs;
                    out.xge[i] = gs + (uint32_t)w - 1u;
                    out.xoff[i] = (int32_t)L;
                    L += w;
                    if (w > 0) {
                        lo = min(lo, gs);
                        hi = max(hi, gs + (uint32_t)w - 1u);
                    }
                }
                if (L == 0 || L > 0x7fffffff) null = true;
            }
        }
        uint32_t clo = 0, chi = 0;
        if (!null) {
            // candidates: start <= span end, and the running max of (end+1) has reached span start
            chi = lower_bound_u32(xs, 0, n_reads, hi + 1u);
            clo = lower_bound_u32(p_maxend1, 0, chi, lo + 1u);
            // NULL rule: at least one (range, read) hit (coverage.R:190-198)
            bool any = false;
            for (uint32_t i = clo; i < chi && !any; i++) {
                const uint32_t rs = xs[i], re1 = p_end1[i];
                if (re1 <= lo) continue;
                const int rst = p_strand ? (int)p_strand[i] : 0;
                for (int64_t q = a; q < b; q++) {
                    const uint32_t s = out.xgs[q], e = out.xge[q];
                    if (e + 1u == s) continue;
                    if (rs <= e && re1 > s &&
                        strand_ok(rst, strand ? (int)strand[q] : 0, ignore_strand, strand_filter)) {
                        any = true;
                        break;
                    }
                }
            }
            if (!any) null = true;
        }
        const int32_t len = null ? 0 : (int32_t)L;
        out.len[g] = len;
        out.flags[g] = (uint8_t)(st0 < 0 ? 1u : 0u);
        out.is_null[g] = null ? 1 : 0;
        out.clo[g] = clo;
        out.chi[g] = chi;
        out.span_lo[g] = lo;
        out.padded[g] = ((int64_t)len + PAD - 1) / PAD * PAD;
        out.ntiles[g] = ((int64_t)len + TILE - 1) / TILE;
        my_null = null ? 1 : 0;
        my_len = (unsigned long long)len;
    }
    unsigned long long my_max = my_len;
    for (int d = 16; d > 0; d >>= 1) {
        my_null += __shfl_xor_sync(0xffffffffu, my_null, d);
        my_len += __shfl_xor_sync(0xffffffffu, my_len, d);
        my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
    }
    if ((threadIdx.x & 31) == 0) {
        if (my_null) atomicAdd(&stats[0], my_null);
        if (my_len) atomicAdd(&stats[1], my_len);
        if (my_max) atomicMax(&stats[2], my_max);
    }
}

// One CTA per (element, tile of the stitched vector).  Every candidate read is tested against
// every range of the element: it contributes `mult` (= number of ranges it overlaps,
// coverage.R:190-192) on each overlapped range, clipped to the tile.
__global__ void __launch_bounds__(CTA)
cov_list_kernel(const int32_t* __restrict__ tile_region, const int64_t* __restrict__ tile_off,
                const int64_t* __restrict__ ptr, const int8_t* __restrict__ strand,
                ListArrays la, const uint32_t* __restrict__ xs,
                const uint32_t* __restrict__ p_end1, const int8_t* __restrict__ p_strand,
                int ignore_strand, int strand_filter, const int64_t* __restrict__ off,
                int32_t* __restrict__ cov) {
    __shared__ __align__(16) int diff[TILE];
    __shared__ int rowpre[MAX_ROWS + 1];
    const int tid = threadIdx.x;
    const int64_t g = tile_region[blockIdx.x];
    const int j = (int)((int64_t)blockIdx.x - tile_off[g]);
    const int L = la.len[g];
    const int m = (L + TILE - 1) / TILE;
    const int tile_len = (((L + m - 1) / m) + ROW - 1) / ROW * ROW;
    const int o_lo = j * tile_len;
    const int tlen = min(tile_len, L - o_lo);
    const bool rev = (la.flags[g] & 1u) != 0;
    const int t0 = rev ? (L - o_lo - tlen) : o_lo;          // stitched offset of the tile
    const int t1 = t0 + tlen - 1;
    const int nrows = (tlen + ROW - 1) / ROW;
    for (int i = tid; i < nrows * (ROW / 4); i += CTA)
        reinterpret_cast<int4*>(diff)[i] = make_int4(0, 0, 0, 0);
    __syncthreads();
    const int64_t a = ptr[g], b = ptr[g + 1];
    const uint32_t clo = la.clo[g], chi = la.chi[g], span_lo = la.span_lo[g];
    for (uint32_t i = clo + tid; i < chi; i += CTA) {
        const uint32_t rs = __ldg(xs + i), re1 = __ldg(p_end1 + i);
        if (re1 <= span_lo) continue;
        const int rst = p_strand ? (int)__ldg(p_strand + i) : 0;
        if (strand_filter != RCP_STRAND_ANY && rst != strand_filter) continue;
        int mult = 0;
        for (int64_t q = a; q < b; q++) {
            const uint32_t s = __ldg(la.xgs + q), e = __ldg(la.xge + q);
            if (e + 1u == s) continue;
            if (rs <= e && re1 > s &&
                strand_ok(rst, strand ? (int)__ldg(strand + q) : 0, ignore_strand, strand_filter))
                mult++;
        }
        if (mult == 0) continue;
        for (int64_t q = a; q < b; q++) {
            const uint32_t s = __ldg(la.xgs + q), e = __ldg(la.xge + q);
            if (e + 1u == s) continue;
            // the selected read covers the chromosome-long vector wherever it lies: every
            // range it touches sees it, hit or not (coverage.R:201-206)
            if (!(rs <= e && re1 > s)) continue;
            const int xo = __ldg(la.xoff + q);
            const int pa = xo + (int)(max(rs, s) - s);
            const int pb = xo + (int)(min(re1 - 1u, e) - s);
            if (pb < t0 || pa > t1) continue;
            // +mult on [max(pa,t0), min(pb,t1)] of the stitched vector, in output order
            const int ka = max(pa, t0) - t0, kb1 = pb + 1 - t0;       // kb1 may equal tlen
            if (!rev) {
                atomicAdd(diff + ka, mult);
                if (kb1 < tlen) atomicSub(diff + kb1, mult);
            } else {
                atomicAdd(diff + (tlen - 1 - ka), mult);
                if (kb1 < tlen) atomicSub(diff + (tlen - 1 - kb1), mult);
            }
        }
    }
    __syncthreads();
    block_scan_store(diff, tlen, 0, rev, rowpre, cov + off[g] + o_lo);
}

// ---- c(left, center, right) -----------------------------------------------------------------
__global__ void __launch_bounds__(CTA)
concat_plan_kernel(int64_t R, const uint8_t* __restrict__ n0, const uint8_t* __restrict__ n1,
                   const uint8_t* __restrict__ n2, const int32_t* __restrict__ l0,
                   const int32_t* __restrict__ l1, const int32_t* __restrict__ l2,
                   int32_t* __restrict__ len, uint8_t* __restrict__ is_null,
                   int64_t* __restrict__ padded, unsigned long long* __restrict__ stats) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= R) return;
    const bool null = n0[r] || n1[r] || n2[r];                    // coverage.R:116-117
    const int64_t L = null ? 0 : (int64_t)l0[r] + l1[r] + l2[r];
    len[r] = (int32_t)L;
    is_null[r] = null ? 1 : 0;
    padded[r] = (L + PAD - 1) / PAD * PAD;
    if (null) {
        atomicAdd(&stats[0], 1ull);
    } else {
        atomicAdd(&stats[1], (unsigned long long)L);
        atomicMax(&stats[2], (unsigned long long)L);
    }
}

__global__ void __launch_bounds__(CTA)
concat_copy_kernel(const int32_t* __restrict__ c0, const int64_t* __restrict__ o0,
                   const int32_t* __restrict__ l0, const int32_t* __restrict__ c1,
                   const int64_t* __restrict__ o1, const int32_t* __restrict__ l1,
                   const int32_t* __restrict__ c2, const int64_t* __restrict__ o2,
                   const int32_t* __restrict__ l2, const int32_t* __restrict__ len,
                   const int64_t* __restrict__ off, int32_t* __restrict__ cov,
                   const unsigned long long* __restrict__ w0, const unsigned long long* __restrict__ w1,
                   const unsigned long long* __restrict__ w2) {
    const int64_t r = blockIdx.x;
    if (len[r] == 0) return;
    int32_t* dst = cov + off[r];
    const int a = l0[r], b = l1[r], c = l2[r];
    const bool n0 = cov_narrow(w0), n1 = cov_narrow(w1), n2 = cov_narrow(w2);
    for (int i = threadIdx.x; i < a; i += CTA) dst[i] = cov_at(c0, o0[r] + i, n0);
    for (int i = threadIdx.x; i < b; i += CTA) dst[a + i] = cov_at(c1, o1[r] + i, n1);
    for (int i = threadIdx.x; i < c; i += CTA) dst[a + b + i] = cov_at(c2, o2[r] + i, n2);
}

__global__ void __launch_bounds__(CTA)
pack_kernel(const int32_t* __restrict__ cov, const int64_t* __restrict__ off,
            const int32_t* __restrict__ len, const int64_t* __restrict__ packed_off,
            int64_t first, int32_t* __restrict__ out, const unsigned long long* __restrict__ bound) {
    const int64_t r = first + blockIdx.x;
    const int L = len[r];
    const bool narrow = cov_narrow(bound);
    const int64_t o = off[r];
    int32_t* dst = out + packed_off[blockIdx.x];
    for (int i = threadIdx.x; i < L; i += CTA) dst[i] = cov_at(cov, o + i, narrow);
}

__global__ void __launch_bounds__(CTA)
len_to_i64_kernel(int64_t n, const int32_t* __restrict__ len, int64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (i < n) out[i] = len[i];
}


// ---- run-length encoding of $coverage (contract T1: one integer Rle per region) ---------------
// runs of region r = #{i : i == 0 or cov[i] != cov[i-1]}
__global__ void __launch_bounds__(CTA)
rle_count_kernel(const int32_t* __restrict__ cov, const int64_t* __restrict__ off,
                 const int32_t* __restrict__ len, int64_t first, int64_t* __restrict__ n_runs,
                 const unsigned long long* __restrict__ bound) {
    __shared__ int wsum[WARPS];
    const int64_t r = first + blockIdx.x;
    const int L = len[r];
    const bool narrow = cov_narrow(bound);
    const int64_t o = off[r];
    int c = 0;
    for (int i = threadIdx.x; i < L; i += CTA)
        c += (i == 0) || (cov_at(cov, o + i, narrow) != cov_at(cov, o + i - 1, narrow));
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < WARPS; w++) t += wsum[w];
        n_runs[blockIdx.x] = t;
    }
}

// values[run] and the start position of every run, region by region (one CTA per region, chunks
// of CTA elements with a running carry)
__global__ void __launch_bounds__(CTA)
rle_write_kernel(const int32_t* __restrict__ cov, const int64_t* __restrict__ off,
                 const int32_t* __restrict__ len, int64_t first,
                 const int64_t* __restrict__ run_ptr, int32_t* __restrict__ values,
                 int32_t* __restrict__ starts, const unsigned long long* __restrict__ bound) {
    __shared__ int wsum[WARPS];
    __shared__ int carry_s;
    const int64_t r = first + blockIdx.x;
    const int L = len[r];
    const bool narrow = cov_narrow(bound);
    const int64_t o = off[r];
    const int64_t base = run_ptr[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int i0 = 0; i0 < L; i0 += CTA) {
        const int i = i0 + threadIdx.x;
        int v = 0;
        bool head = false;
        if (i < L) {
            v = cov_at(cov, o + i, narrow);
            head = (i == 0) || (v != cov_at(cov, o + i - 1, narrow));
        }
        const unsigned bal = __ballot_sync(0xffffffffu, head);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int pre = carry_s;
        for (int w = 0; w < warp; w++) pre += wsum[w];
        if (head) {
            const int64_t o = base + pre + __popc(bal & ((1u << lane) - 1u));
            values[o] = v;
            starts[o] = i;
        }
        __syncthreads();
        if (threadIdx.x == CTA - 1) carry_s = pre + __popc(bal);
        __syncthreads();
    }
}

// lengths[run] = start of the next run of the same region (or the region length) - start
__global__ void __launch_bounds__(CTA)
rle_lengths_kernel(const int32_t* __restrict__ len, int64_t first,
                   const int64_t* __restrict__ run_ptr, const int32_t* __restrict__ starts,
                   int32_t* __restrict__ lengths) {
    const int64_t r = first + blockIdx.x;
    const int L = len[r];
    const int64_t a = run_ptr[blockIdx.x], b = run_ptr[blockIdx.x + 1];
    for (int64_t j = a + threadIdx.x; j < b; j += CTA)
        lengths[j] = (j + 1 < b ? starts[j + 1] : L) - starts[j];
}

int alloc_coverage_arrays(Coverage* cv, int64_t R) {
    cv->n_regions = R;
    RCP_TRY(dalloc(&cv->off, (size_t)R + 1));
    RCP_TRY(dalloc(&cv->len, (size_t)R));
    RCP_TRY(dalloc(&cv->is_null, (size_t)R));
    return RCP_OK;
}

template <int NS>
int coverage_ranges_impl(ReadsIdx& rd, Sources<NS> src, int64_t R, const int32_t* chrom,
                         const int32_t* start, const int32_t* end, const int8_t* strand,
                         int ignore_strand, int strand_filter, Coverage* cv) {
    RCP_TRY(alloc_coverage_arrays(cv, R));
    RegionArrays ra;
    RCP_TRY(dalloc(&ra.gs, (size_t)R));
    ra.len = cv->len;
    RCP_TRY(dalloc(&ra.flags, (size_t)R));
    ra.is_null = cv->is_null;
    RCP_TRY(dalloc(&ra.ix0, (size_t)R * NS));
    RCP_TRY(dalloc(&ra.ix1, (size_t)R * NS));
    RCP_TRY(dalloc(&ra.iy0, (size_t)R * NS));
    RCP_TRY(dalloc(&ra.iy1, (size_t)R * NS));
    RCP_TRY(dalloc(&ra.padded, (size_t)R));
    RCP_TRY(dalloc(&ra.ntiles, (size_t)R));
    int64_t* tile_off = nullptr;
    RCP_TRY(dalloc(&tile_off, (size_t)R + 1));
    unsigned int* d_err = nullptr;
    unsigned long long* d_stats = nullptr;
    RCP_TRY(dalloc(&d_err, 1));
    RCP_TRY(dalloc(&d_stats, 3));
    RCP_CUDA(cudaMemsetAsync(d_err, 0, sizeof(unsigned int), g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(d_stats, 0, 3 * sizeof(unsigned long long), g_ctx.stream));

    struct Host {
        int64_t total_padded, total_tiles;
        unsigned long long stats[3];
        unsigned int err;
    } h = {0, 0, {0, 0, 0}, 0};
    {
        StageTimer t(ST_COV_PLAN);
        if (R > 0) {
            region_plan_kernel<NS><<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(
                R, chrom, start, end, strand, rd.d_chrom_off, rd.d_chrom_len, rd.n_chrom, src,
                ignore_strand, strand_filter, ra, d_err, d_stats);
            RCP_LAUNCHED();
        }
        RCP_TRY(exclusive_scan2_i64(ra.padded, cv->off, cv->off + R, ra.ntiles, tile_off,
                                    tile_off + R, R));
    }
    {
        const FetchItem items[4] = {{cv->off + R, &h.total_padded, 8}, {tile_off + R, &h.total_tiles, 8},
                                    {d_stats, h.stats, 24}, {d_err, &h.err, 4}};
        RCP_TRY(fetch_and_sync(items, 4));
    }
    int rc = RCP_OK;
    if (h.err & 1u) rc = fail(RCP_ERR_DATA, "a region has a chromosome id outside [0, n_chrom)");
    else if (h.err & 2u) rc = fail(RCP_ERR_DATA, "a region has end < start - 1");
    if (rc == RCP_OK) {
        cv->path = RCP_PATH_INDEX;
        cv->total_padded = h.total_padded;
        cv->n_null = (int64_t)h.stats[0];
        cv->total_len = (int64_t)h.stats[1];
        cv->max_len = (int32_t)h.stats[2];
        rc = dalloc(&cv->cov, (size_t)h.total_padded);
    }
    int32_t* tile_region = nullptr;
    if (rc == RCP_OK && h.total_tiles > 0) {
        rc = dalloc(&tile_region, (size_t)h.total_tiles);
        if (rc == RCP_OK) {
            {
                StageTimer t(ST_COV_PLAN);
                fill_tiles_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(R, ra.ntiles,
                                                                                tile_off, tile_region);
                g_ctx.launches++;
            }
            StageTimer t(ST_COV_TILE);
            cov_tile_kernel<NS><<<(unsigned)h.total_tiles, CTA, 0, g_ctx.stream>>>(
                tile_region, tile_off, ra, src, cv->off, cv->cov);
            g_ctx.launches++;
        }
    }
    if (rc == RCP_OK && R > 0) {
        StageTimer t(ST_COV_SMALL);
        cov_small_kernel<NS><<<blocks_for(R, WARPS), CTA, 0, g_ctx.stream>>>(R, ra, src, cv->off,
                                                                             cv->cov);
        g_ctx.launches++;
    }
    if (rc == RCP_OK && cudaGetLastError() != cudaSuccess)
        rc = fail(RCP_ERR_CUDA, "coverage kernel launch failed");
    dfree(tile_region);
    dfree(ra.gs);
    dfree(ra.flags);
    dfree(ra.ix0);
    dfree(ra.ix1);
    dfree(ra.iy0);
    dfree(ra.iy1);
    dfree(ra.padded);
    dfree(ra.ntiles);
    dfree(tile_off);
    dfree(d_err);
    dfree(d_stats);
    return rc;
}

}  // namespace

void coverage_release(Coverage& c) {
    dfree(c.cov);
    dfree(c.off);
    dfree(c.len);
    dfree(c.is_null);
    dfree(c.d_stats);
    c.d_bound = nullptr;
    c.stats_pending = false;
}

// ---- NA seqlengths (coverage.R:201) ----------------------------------------------------------
// coverage(y$reads)[[chr]] of a chromosome of unknown length ends at the largest end among the
// reads that OVERLAP the region, and indexing beyond it is the "invalid genomic area" error ->
// NULL (coverage.R:206-209,217-222).  A read that overlaps the region and ends at or after the
// region's last position covers that position, so the rule reads: NULL unless the coverage at the
// region's genomic end is non-zero.
namespace {
__global__ void __launch_bounds__(CTA)
na_rule_kernel(int64_t R, const int32_t* __restrict__ chrom, const int8_t* __restrict__ strand,
               const uint8_t* __restrict__ len_na, int n_chrom, const int64_t* __restrict__ off,
               int32_t* __restrict__ len, uint8_t* __restrict__ is_null, const int32_t* __restrict__ cov,
               const int64_t* __restrict__ end_pos, const unsigned long long* __restrict__ bound) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= R) return;
    const int32_t L = len[r];
    const int c = chrom[r];
    if (L <= 0 || c < 0 || c >= n_chrom || !len_na[c]) return;
    const int64_t idx = end_pos ? end_pos[r] : ((strand && strand[r] < 0) ? 0 : (int64_t)L - 1);
    if (idx < 0 || idx >= L || cov_at(cov, off[r] + idx, cov_narrow(bound)) == 0) {
        len[r] = 0;
        is_null[r] = 1;
    }
}

__global__ void __launch_bounds__(CTA)
len_stats_kernel(int64_t R, const int32_t* __restrict__ len, unsigned long long* __restrict__ stats) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (r < R) {
        my_len = (unsigned long long)len[r];
        my_null = my_len == 0 ? 1 : 0;
    }
    unsigned long long my_max = my_len;
    for (int d = 16; d > 0; d >>= 1) {
        my_null += __shfl_xor_sync(0xffffffffu, my_null, d);
        my_len += __shfl_xor_sync(0xffffffffu, my_len, d);
        my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
    }
    if ((threadIdx.x & 31) == 0) {
        if (my_null) atomicAdd(&stats[0], my_null);
        if (my_len) atomicAdd(&stats[1], my_len);
        if (my_max) atomicMax(&stats[2], my_max);
    }
}
}  // namespace

int coverage_na_rule(const ReadsIdx& rd, Coverage& cv, int64_t R, const int32_t* d_chrom, const int8_t* d_strand,
                     const int64_t* d_end_pos) {
    if (!rd.any_na || R <= 0) return RCP_OK;
    RCP_TRY(coverage_resolve_stats(cv));            // (keeps `candidates`; the rest is recomputed)
    if (!cv.d_stats) RCP_TRY(dalloc(&cv.d_stats, 4));
    const unsigned long long h[4] = {0ull, 0ull, 0ull, (unsigned long long)cv.candidates};
    RCP_CUDA(cudaMemcpyAsync(cv.d_stats, h, 32, cudaMemcpyHostToDevice, g_ctx.stream));
    na_rule_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(R, d_chrom, d_strand, rd.d_len_na, rd.n_chrom, cv.off,
                                                               cv.len, cv.is_null, cv.cov, d_end_pos, cv.d_bound);
    RCP_LAUNCHED();
    len_stats_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(R, cv.len, cv.d_stats);
    RCP_LAUNCHED();
    cv.stats_pending = true;
    return coverage_resolve_stats(cv);
}

// split path: n_null / total_len / max_len / candidates were produced after the call returned
int coverage_resolve_stats(Coverage& c) {
    if (!c.stats_pending) return RCP_OK;
    unsigned long long h[4] = {0, 0, 0, 0};
    const FetchItem items[1] = {{c.d_stats, h, 32}};
    RCP_TRY(fetch_and_sync(items, 1));
    c.n_null = (int64_t)h[0];
    c.total_len = (int64_t)h[1];
    c.max_len = (int32_t)h[2];
    c.candidates = (int64_t)h[3];
    c.stats_pending = false;
    return RCP_OK;
}

int coverage_ranges(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                    const int32_t* end, const int8_t* strand, int ignore_strand,
                    int strand_filter, int mem, Coverage* cv) {
    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_chrom.init(chrom, (size_t)R, mem));
    RCP_TRY(d_start.init(start, (size_t)R, mem));
    RCP_TRY(d_end.init(end, (size_t)R, mem));
    RCP_TRY(d_strand.init(strand, (size_t)R, mem));
    const bool unstranded = (strand_filter == RCP_STRAND_ANY) && (ignore_strand || strand == nullptr);
    const bool uni = rd.uniform_w != 0;
    auto fill = [&](auto& src, int slot, int cls, int bit) {
        const SortedClass& sc = rd.cls[cls];
        src.xs[slot] = sc.xs;
        src.ye[slot] = uni ? sc.xs : sc.ye;
        src.yshift[slot] = rd.uniform_w;
        src.n[slot] = (uint32_t)sc.n;
        src.cls_bit[slot] = (uint8_t)bit;
        src.corr[slot] = 0;
    };
    auto fill_corr = [&](auto& src, int slot, int cls, int bit) {
        const SortedClass& sc = rd.cls[cls];
        src.xs[slot] = sc.cxs;
        src.ye[slot] = sc.cye;
        src.yshift[slot] = 0;
        src.n[slot] = (uint32_t)sc.cn;
        src.cls_bit[slot] = (uint8_t)bit;
        src.corr[slot] = 1;
    };
    if (unstranded) {
        RCP_TRY(reads_build_class(rd, CLS_ALL));
        if (!uni) {
            Sources<1> src;
            fill(src, 0, CLS_ALL, 0);
            return coverage_ranges_impl<1>(rd, src, R, d_chrom.ptr, d_start.ptr, d_end.ptr,
                                           d_strand.ptr, ignore_strand, strand_filter, cv);
        }
        Sources<2> src;
        fill(src, 0, CLS_ALL, 0);
        fill_corr(src, 1, CLS_ALL, 0);
        return coverage_ranges_impl<2>(rd, src, R, d_chrom.ptr, d_start.ptr, d_end.ptr,
                                       d_strand.ptr, ignore_strand, strand_filter, cv);
    }
    for (int k = 0; k < 3; k++) RCP_TRY(reads_build_class(rd, CLS_PLUS + k));
    if (!uni) {
        Sources<3> src;
        for (int k = 0; k < 3; k++) fill(src, k, CLS_PLUS + k, k);
        return coverage_ranges_impl<3>(rd, src, R, d_chrom.ptr, d_start.ptr, d_end.ptr,
                                       d_strand.ptr, ignore_strand, strand_filter, cv);
    }
    Sources<6> src;
    for (int k = 0; k < 3; k++) {
        fill(src, k, CLS_PLUS + k, k);
        fill_corr(src, 3 + k, CLS_PLUS + k, k);
    }
    return coverage_ranges_impl<6>(rd, src, R, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr,
                                   ignore_strand, strand_filter, cv);
}

int coverage_list(ReadsIdx& rd, int64_t G, const int64_t* ptr, const int64_t n_ranges,
                  const int32_t* chrom, const int32_t* start, const int32_t* end,
                  const int8_t* strand, int ignore_strand, int strand_filter, int mem,
                  Coverage* cv) {
    RCP_TRY(reads_build_pairs(rd));
    DevIn<int64_t> d_ptr;
    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_ptr.init(ptr, (size_t)G + 1, mem));
    RCP_TRY(d_chrom.init(chrom, (size_t)n_ranges, mem));
    RCP_TRY(d_start.init(start, (size_t)n_ranges, mem));
    RCP_TRY(d_end.init(end, (size_t)n_ranges, mem));
    RCP_TRY(d_strand.init(strand, (size_t)n_ranges, mem));
    RCP_TRY(alloc_coverage_arrays(cv, G));
    ListArrays la;
    RCP_TRY(dalloc(&la.xgs, (size_t)n_ranges));
    RCP_TRY(dalloc(&la.xge, (size_t)n_ranges));
    RCP_TRY(dalloc(&la.xoff, (size_t)n_ranges));
    la.len = cv->len;
    la.is_null = cv->is_null;
    RCP_TRY(dalloc(&la.flags, (size_t)G));
    RCP_TRY(dalloc(&la.clo, (size_t)G));
    RCP_TRY(dalloc(&la.chi, (size_t)G));
    RCP_TRY(dalloc(&la.span_lo, (size_t)G));
    RCP_TRY(dalloc(&la.padded, (size_t)G));
    RCP_TRY(dalloc(&la.ntiles, (size_t)G));
    int64_t* tile_off = nullptr;
    RCP_TRY(dalloc(&tile_off, (size_t)G + 1));
    unsigned int* d_err = nullptr;
    unsigned long long* d_stats = nullptr;
    RCP_TRY(dalloc(&d_err, 1));
    RCP_TRY(dalloc(&d_stats, 3));
    RCP_CUDA(cudaMemsetAsync(d_err, 0, sizeof(unsigned int), g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(d_stats, 0, 3 * sizeof(unsigned long long), g_ctx.stream));
    struct Host {
        int64_t total_padded, total_tiles;
        unsigned long long stats[3];
        unsigned int err;
    } h = {0, 0, {0, 0, 0}, 0};
    StageTimer list_timer(ST_COV_LIST);
    if (G > 0) {
        list_plan_kernel<<<blocks_for(G, CTA), CTA, 0, g_ctx.stream>>>(
            G, d_ptr.ptr, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr, rd.d_chrom_off,
            rd.d_chrom_len, rd.n_chrom, rd.cls[CLS_ALL].xs, rd.p_end1, rd.p_strand, rd.p_maxend1,
            (uint32_t)rd.n, ignore_strand, strand_filter, la, d_err, d_stats);
        RCP_LAUNCHED();
    }
    RCP_TRY(exclusive_scan2_i64(la.padded, cv->off, cv->off + G, la.ntiles, tile_off,
                                tile_off + G, G));
    {
        const FetchItem items[4] = {{cv->off + G, &h.total_padded, 8}, {tile_off + G, &h.total_tiles, 8},
                                    {d_stats, h.stats, 24}, {d_err, &h.err, 4}};
        RCP_TRY(fetch_and_sync(items, 4));
    }
    int rc = RCP_OK;
    if (h.err & 1u) rc = fail(RCP_ERR_DATA, "a range has a chromosome id outside [0, n_chrom)");
    else if (h.err & 2u) rc = fail(RCP_ERR_DATA, "a range has end < start - 1");
    else if (h.err & 4u)
        rc = fail(RCP_ERR_DATA, "the ranges of one list element lie on different chromosomes");
    if (rc == RCP_OK) {
        cv->total_padded = h.total_padded;
        cv->n_null = (int64_t)h.stats[0];
        cv->total_len = (int64_t)h.stats[1];
        cv->max_len = (int32_t)h.stats[2];
        rc = dalloc(&cv->cov, (size_t)h.total_padded);
    }
    int32_t* tile_region = nullptr;
    if (rc == RCP_OK && h.total_tiles > 0) {
        rc = dalloc(&tile_region, (size_t)h.total_tiles);
        if (rc == RCP_OK) {
            fill_tiles_kernel<<<blocks_for(G, CTA), CTA, 0, g_ctx.stream>>>(G, la.ntiles, tile_off,
                                                                            tile_region);
            g_ctx.launches++;
            cov_list_kernel<<<(unsigned)h.total_tiles, CTA, 0, g_ctx.stream>>>(
                tile_region, tile_off, d_ptr.ptr, d_strand.ptr, la, rd.cls[CLS_ALL].xs, rd.p_end1,
                rd.p_strand, ignore_strand, strand_filter, cv->off, cv->cov);
            g_ctx.launches++;
            if (cudaGetLastError() != cudaSuccess)
                rc = fail(RCP_ERR_CUDA, "list coverage kernel launch failed");
        }
    }
    dfree(tile_region);
    dfree(la.xgs);
    dfree(la.xge);
    dfree(la.xoff);
    dfree(la.flags);
    dfree(la.clo);
    dfree(la.chi);
    dfree(la.span_lo);
    dfree(la.padded);
    dfree(la.ntiles);
    dfree(tile_off);
    dfree(d_err);
    dfree(d_stats);
    return rc;
}

int coverage_concat3(const Coverage& a, const Coverage& b, const Coverage& c, Coverage* cv) {
    const int64_t R = a.n_regions;
    if (b.n_regions != R || c.n_regions != R)
        return fail(RCP_ERR_ARG, "concat3: the three coverages have different lengths");
    RCP_TRY(alloc_coverage_arrays(cv, R));
    int64_t* padded = nullptr;
    unsigned long long* d_stats = nullptr;
    RCP_TRY(dalloc(&padded, (size_t)R));
    RCP_TRY(dalloc(&d_stats, 3));
    RCP_CUDA(cudaMemsetAsync(d_stats, 0, 24, g_ctx.stream));
    if (R > 0) {
        concat_plan_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(
            R, a.is_null, b.is_null, c.is_null, a.len, b.len, c.len, cv->len, cv->is_null, padded,
            d_stats);
        RCP_LAUNCHED();
    }
    RCP_TRY(exclusive_scan_i64(padded, cv->off, R, cv->off + R));
    int64_t total = 0;
    unsigned long long stats[3] = {0, 0, 0};
    StageTimer concat_timer(ST_COV_CONCAT);
    RCP_CUDA(cudaMemcpyAsync(&total, cv->off + R, 8, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(stats, d_stats, 24, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    cv->total_padded = total;
    cv->n_null = (int64_t)stats[0];
    cv->total_len = (int64_t)stats[1];
    cv->max_len = (int32_t)stats[2];
    RCP_TRY(dalloc(&cv->cov, (size_t)total));
    if (R > 0) {
        concat_copy_kernel<<<(unsigned)R, CTA, 0, g_ctx.stream>>>(a.cov, a.off, a.len, b.cov, b.off,
                                                                 b.len, c.cov, c.off, c.len,
                                                                 cv->len, cv->off, cv->cov, a.d_bound,
                                                                 b.d_bound, c.d_bound);
        RCP_LAUNCHED();
    }
    dfree(padded);
    dfree(d_stats);
    return RCP_OK;
}

int coverage_fetch(const Coverage& cv, int64_t first, int64_t count, int32_t* out,
                   int64_t capacity) {
    if (first < 0 || count < 0 || first + count > cv.n_regions)
        return fail(RCP_ERR_ARG, "fetch: region range [%lld, %lld) outside [0, %lld)",
                    (long long)first, (long long)(first + count), (long long)cv.n_regions);
    if (count == 0) return RCP_OK;
    int64_t *len64 = nullptr, *poff = nullptr;
    RCP_TRY(dalloc(&len64, (size_t)count));
    RCP_TRY(dalloc(&poff, (size_t)count + 1));
    len_to_i64_kernel<<<blocks_for(count, CTA), CTA, 0, g_ctx.stream>>>(count, cv.len + first, len64);
    RCP_LAUNCHED();
    RCP_TRY(exclusive_scan_i64(len64, poff, count, poff + count));
    int64_t total = 0;
    RCP_CUDA(cudaMemcpyAsync(&total, poff + count, 8, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    int rc = RCP_OK;
    if (total > capacity) {
        rc = fail(RCP_ERR_ARG, "fetch: %lld ints needed, capacity %lld", (long long)total,
                  (long long)capacity);
    } else if (total > 0) {
        int32_t* packed = nullptr;
        rc = dalloc(&packed, (size_t)total);
        if (rc == RCP_OK) {
            pack_kernel<<<(unsigned)count, CTA, 0, g_ctx.stream>>>(cv.cov, cv.off, cv.len, poff,
                                                                  first, packed, cv.d_bound);
            g_ctx.launches++;
            cudaError_t e = cudaMemcpyAsync(out, packed, (size_t)total * 4, cudaMemcpyDeviceToHost,
                                            g_ctx.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "fetch copy failed: %s", cudaGetErrorString(e));
            dfree(packed);
        }
    }
    dfree(len64);
    dfree(poff);
    return rc;
}

// Run-length encoding of regions [first, first + count): run_ptr (count + 1, host) receives the
// offsets of each region's runs; values / lengths (host, `capacity` entries each, may be null to
// only count) receive the runs.  NULL regions have no runs.
int coverage_rle(const Coverage& cv, int64_t first, int64_t count, int64_t* run_ptr,
                 int32_t* values, int32_t* lengths, int64_t capacity) {
    if (first < 0 || count < 0 || first + count > cv.n_regions)
        return fail(RCP_ERR_ARG, "rle: region range [%lld, %lld) outside [0, %lld)", (long long)first,
                    (long long)(first + count), (long long)cv.n_regions);
    if (run_ptr == nullptr) return fail(RCP_ERR_ARG, "rle: run_ptr is NULL");
    run_ptr[0] = 0;
    if (count == 0) return RCP_OK;
    int64_t *n_runs = nullptr, *d_ptr = nullptr;
    RCP_TRY(dalloc(&n_runs, (size_t)count));
    RCP_TRY(dalloc(&d_ptr, (size_t)count + 1));
    rle_count_kernel<<<(unsigned)count, CTA, 0, g_ctx.stream>>>(cv.cov, cv.off, cv.len, first, n_runs, cv.d_bound);
    RCP_LAUNCHED();
    RCP_TRY(exclusive_scan_i64(n_runs, d_ptr, count, d_ptr + count));
    RCP_CUDA(cudaMemcpyAsync(run_ptr, d_ptr, ((size_t)count + 1) * 8, cudaMemcpyDeviceToHost,
                             g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    const int64_t total = run_ptr[count];
    int rc = RCP_OK;
    if (values != nullptr || lengths != nullptr) {
        if (values == nullptr || lengths == nullptr)
            rc = fail(RCP_ERR_ARG, "rle: values and lengths must be given together");
        else if (total > capacity)
            rc = fail(RCP_ERR_ARG, "rle: %lld runs, capacity %lld", (long long)total, (long long)capacity);
        else if (total > 0) {
            int32_t *d_val = nullptr, *d_start = nullptr, *d_len = nullptr;
            rc = dalloc(&d_val, (size_t)total);
            if (rc == RCP_OK) rc = dalloc(&d_start, (size_t)total);
            if (rc == RCP_OK) rc = dalloc(&d_len, (size_t)total);
            if (rc == RCP_OK) {
                rle_write_kernel<<<(unsigned)count, CTA, 0, g_ctx.stream>>>(cv.cov, cv.off, cv.len, first,
                                                                           d_ptr, d_val, d_start, cv.d_bound);
                g_ctx.launches++;
                rle_lengths_kernel<<<(unsigned)count, CTA, 0, g_ctx.stream>>>(cv.len, first, d_ptr,
                                                                             d_start, d_len);
                g_ctx.launches++;
                cudaError_t e = cudaMemcpyAsync(values, d_val, (size_t)total * 4, cudaMemcpyDeviceToHost,
                                                g_ctx.stream);
                if (e == cudaSuccess)
                    e = cudaMemcpyAsync(lengths, d_len, (size_t)total * 4, cudaMemcpyDeviceToHost,
                                        g_ctx.stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
                if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "rle copy failed: %s", cudaGetErrorString(e));
            }
            dfree(d_val);
            dfree(d_start);
            dfree(d_len);
        }
    }
    dfree(n_runs);
    dfree(d_ptr);
    return rc;
}

}  // namespace rcp
