// Device helpers shared by the coverage kernels (coverage.cu: sorted-index path and
// GRangesList path; coverage_buckets.cu: reads bucketed per output tile, no sort;
// coverage_split.cu: the one-pass split path).
#pragma once
#include "rcp_internal.cuh"

namespace rcp {
namespace covk {

constexpr int CTA = 256;
constexpr int WARPS = CTA / 32;
constexpr int TILE = 7168;             // positions per CTA tile (28 KB of int32; 8 CTAs per SM)
constexpr int ROW = 128;               // positions handled by one warp-wide int4 access
constexpr int MAX_ROWS = TILE / ROW;   // 56
static_assert(MAX_ROWS == 7 * WARPS, "tile kernels dispatch on 1..7 rows per warp");
constexpr int SMALL_MAX = 1024;        // regions up to this length use the warp kernel
constexpr int PAD = 32;                // region offsets are multiples of 32 ints (128 B)


// classes (bit0 '+', bit1 '-', bit2 '*') a region may count under the strand rules of
// calcCoverage(strand=) (coverage.R:141-144) and findOverlaps(ignore.strand=) (coverage.R:191)
__device__ __forceinline__ unsigned class_mask(int region_strand, int ignore_strand,
                                               int strand_filter) {
    unsigned m = 7u;
    if (strand_filter != RCP_STRAND_ANY) m = strand_filter > 0 ? 1u : (strand_filter < 0 ? 2u : 4u);
    if (!ignore_strand) {
        if (region_strand > 0) m &= 5u;
        else if (region_strand < 0) m &= 6u;
    }
    return m;
}

// Window geometry of one region (coverage.R:209 inside the tryCatch of coverage.R:217-222):
// `[start:end]` on the chromosome-long vector -- a negative start mixes signs, an end past the
// chromosome is out of bounds -> NULL; a zero index is silently dropped.  Returns true when the
// region is NULL for geometric reasons; *gs = global coordinate of the first base, *L = length.
// err bits: 1 chrom id out of range, 2 end < start - 1.
__device__ __forceinline__ bool window_geometry(int c, int64_t s, int64_t e, int n_chrom,
                                                const uint32_t* __restrict__ chrom_off,
                                                const int64_t* __restrict__ chrom_len,
                                                unsigned int* __restrict__ err, uint32_t* gs,
                                                int64_t* L) {
    *gs = 0;
    *L = 0;
    if (c < 0 || c >= n_chrom) {
        atomicOr(err, 1u);
        return true;
    }
    if (e < s - 1) {
        atomicOr(err, 2u);
        return true;
    }
    bool null = false;
    if (s < 0 || e > chrom_len[c]) null = true;
    if (s == 0) s = 1;
    int64_t len = e - s + 1;
    if (len <= 0) { len = 0; null = true; }
    *L = len;
    *gs = chrom_off[c] + (uint32_t)(s > 0 ? s : 0);
    return null;
}

__device__ __forceinline__ bool strand_ok(int read_strand, int range_strand, int ignore_strand,
                                          int strand_filter) {
    if (strand_filter != RCP_STRAND_ANY && read_strand != strand_filter) return false;
    if (ignore_strand || range_strand == 0 || read_strand == 0) return true;
    return read_strand == range_strand;
}


// --------------------------------------------------------------------------------------------
// Scan + store.  `diff` holds the tile's difference array IN OUTPUT ORDER: for a '-' region the
// events are scattered mirrored (index tlen-1-k), so the output is always written left to right
// with aligned 16-byte stores straight from registers:
//     '+'  out[k] = base + inclusive_prefix(k)
//     '-'  out[k] = base + total - exclusive_prefix(k)        (a suffix sum of the mirrored array)
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_inclusive_scan(int v) {
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += o;
    }
    return v;
}

// One row (128 outputs at dst[0..127], `valid` of them real) by one warp.  `pre` = sum of every
// diff before this row.  Returns the row total (all lanes).
__device__ __forceinline__ int warp_row_scan_store(const int* row_ptr, int pre, int base_or_top,
                                                   bool rev, int valid, int32_t* __restrict__ dst) {
    const int lane = threadIdx.x & 31;
    const int4 v = *(reinterpret_cast<const int4*>(row_ptr) + lane);
    const int i0 = v.x, i1 = i0 + v.y, i2 = i1 + v.z, i3 = i2 + v.w;
    const int inc = warp_inclusive_scan(i3);
    const int ex = pre + inc - i3;                 // sum of everything before this lane's 4
    int4 o;
    if (!rev) {
        o = make_int4(base_or_top + ex + i0, base_or_top + ex + i1, base_or_top + ex + i2,
                      base_or_top + ex + i3);
    } else {
        o = make_int4(base_or_top - ex, base_or_top - ex - i0, base_or_top - ex - i1,
                      base_or_top - ex - i2);
    }
    const int k = lane * 4;
    if (k + 3 < valid) {
        *reinterpret_cast<int4*>(dst + k) = o;
    } else {
        if (k < valid) dst[k] = o.x;
        if (k + 1 < valid) dst[k + 1] = o.y;
        if (k + 2 < valid) dst[k + 2] = o.z;
    }
    return __shfl_sync(0xffffffffu, inc, 31);
}

// Whole CTA: tile of `tlen` outputs at dst (16-byte aligned).  rowpre needs MAX_ROWS + 1 ints.
__device__ __forceinline__ void block_scan_store(const int* diff, int tlen, int base, bool rev,
                                                 int* rowpre, int32_t* __restrict__ dst) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nrows = (tlen + ROW - 1) / ROW;
    for (int row = warp; row < nrows; row += WARPS) {          // pass A: row totals
        const int4 v = *(reinterpret_cast<const int4*>(diff + row * ROW) + lane);
        int s = v.x + v.y + v.z + v.w;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (lane == 0) rowpre[row] = s;
    }
    __syncthreads();
    if (warp == 0) {                                           // exclusive prefix of the rows
        int carry = 0;
        for (int r0 = 0; r0 < nrows; r0 += 32) {
            const int r = r0 + lane;
            const int v = r < nrows ? rowpre[r] : 0;
            const int inc = warp_inclusive_scan(v);
            if (r < nrows) rowpre[r] = carry + inc - v;
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) rowpre[MAX_ROWS] = carry;               // tile total
    }
    __syncthreads();
    const int top = rev ? base + rowpre[MAX_ROWS] : base;
    for (int row = warp; row < nrows; row += WARPS)            // pass B: scan + store
        warp_row_scan_store(diff + row * ROW, rowpre[row], top, rev, tlen - row * ROW,
                            dst + row * ROW);
}

// --------------------------------------------------------------------------------------------
// Forward scan + store, lane-serial (bucket path: '-' regions are mirrored when the events are
// written, so the tile kernels only ever scan forwards).  A warp owns RPW consecutive rows
// (RPW * 128 ints); lane l owns the RPW * 4 consecutive ints at l * RPW * 4 of them (16-byte
// loads with a lane stride of RPW * 16 bytes: conflict-free for odd RPW).  The lane sums its
// run, one warp scan orders the lanes, the run is rescanned from the right start and written
// back in place; the warp then streams its rows out with aligned 16-byte stores.  About a
// third of the instructions of the row-by-row scan above (one shuffle scan per RPW * 128
// outputs instead of per 128).
// --------------------------------------------------------------------------------------------
// ---- TMA 1-D bulk store (shared -> global), bulk-group completion ------------------------------
__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(gmem_dst), "r"((uint32_t)__cvta_generic_to_shared(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// the bulk stores issued by this thread have finished READING shared memory
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// rows [row0, row0 + RPW) of the scanned tile -> dst, fully unrolled
template <int RPW>
__device__ __forceinline__ void warp_rows_out_n(const int* tile, int row0, int tlen,
                                                int32_t* __restrict__ dst) {
    const int lane = threadIdx.x & 31;
    const int base = row0 * ROW + lane * 4;
    const int* src = tile + base;
    int32_t* out = dst + base;
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        const int o0 = base + k * ROW;
        if (o0 + 3 < tlen) {
            *reinterpret_cast<int4*>(out + k * ROW) = *reinterpret_cast<const int4*>(src + k * ROW);
        } else if (o0 < tlen) {
            const int4 o = *reinterpret_cast<const int4*>(src + k * ROW);
            out[k * ROW] = o.x;
            if (o0 + 1 < tlen) out[k * ROW + 1] = o.y;
            if (o0 + 2 < tlen) out[k * ROW + 2] = o.z;
        }
    }
}

// Whole CTA, RPW rows per warp (compile-time: every loop unrolls, no predicates).  `diff` must be
// zero-padded up to WARPS * RPW rows.  wtot needs WARPS ints.
template <int RPW, bool TMA_OUT>
__device__ __forceinline__ void block_scan_store_fwd(int* diff, int tlen, int* wtot,
                                                     int32_t* __restrict__ dst) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* mine = diff + (warp * ROW + lane * 4) * RPW;
    int4 v[RPW];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        v[k] = *(reinterpret_cast<const int4*>(mine) + k);
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
    const int inc = warp_inclusive_scan(sum);
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    int run = inc - sum;
#pragma unroll
    for (int w = 0; w < WARPS - 1; w++)
        if (w < warp) run += wtot[w];
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        int4 o;
        o.x = (run += v[k].x);
        o.y = (run += v[k].y);
        o.z = (run += v[k].z);
        o.w = (run += v[k].w);
        *(reinterpret_cast<int4*>(mine) + k) = o;
    }
    __syncwarp();
    if (TMA_OUT) {
        // the warp's rows are contiguous in shared memory and in the output: one bulk store by
        // the TMA unit (16-byte granules; a ragged tail spills <= 3 ints into the region's own
        // padding).  The caller waits for the store to have read shared memory
        // (tma_store_wait_read) before the tile buffer is reused.
        if (lane == 0) {
            const int c0 = warp * RPW * ROW;
            const int valid = min(RPW * ROW, tlen - c0);
            if (valid > 0) {
                fence_proxy_async_smem();
                tma_store_1d(dst + c0, diff + c0, (uint32_t)((valid + 3) & ~3) * 4u);
                tma_store_commit();
            }
        }
    } else {
        warp_rows_out_n<RPW>(diff, warp * RPW, tlen, dst);
    }
}

inline unsigned blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

}  // namespace covk
}  // namespace rcp
