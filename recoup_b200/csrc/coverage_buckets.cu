// Coverage without a sort (sm_100a): calcCoverage / coverageFromRanges of the reference
// (/root/reference/R/coverage.R:126-226) straight from the UNSORTED reads: the BUCKET path
// (bkt_*).  RCP_PATH_AUTO takes it for GRanges masks whose reads are too wide for the split path
// (coverage_split.cu); the scan / store code of its tiles is shared (cov_common.cuh).
//
// Only reads that overlap a region contribute to that region's coverage, and a region's coverage
// does not depend on the order of its reads.  So instead of sorting every read by coordinate
// (index.cu + sort.cu) this path drops each read into the buckets of the OUTPUT TILES it
// overlaps -- the region-sorted read lists the coverage kernels consume:
//
//   1. plan          regions -> windows (geometry / NULL rules) -> tiles (<= 7168 outputs, cut
//                    in output space; regions <= 1024 bp are one warp-sized tile)
//   2. cell table    the genome is cut into 2048-bp cells; one 16-byte record per cell holds
//                    the first tile overlapping it inline (L2-resident), further tiles in
//                    overflow runs
//   3. find pass     every read is checked against a shared-memory bitmap of the 16-kb blocks
//                    some tile touches (most reads of a sparse mask stop there), then against
//                    the 16-byte record of each cell it touches; a hit is clipped to the tile,
//                    packed as ONE 32-bit event pair (first covered output | one past the last;
//                    '-' regions are mirrored here, so the tile kernels are strand-agnostic),
//                    appended to a hit list and counted per tile
//   4. NULL rule     a region with no read in any tile is NULL (coverage.R:198,224-225);
//                    offsets of the dense coverage and of the buckets by prefix sums
//   5. place pass    hit list -> per-tile buckets (a counting sort by tile)
//   6. tile kernels  bucket -> shared-memory difference array (atomics) -> block prefix scan ->
//                    aligned 16-byte stores of the int32 coverage
//
// HBM traffic: 8-9 B per read once + 20 B per (read, tile) hit, against >= 4 passes x 8 B per
// read for a radix sort of the whole read set.
#include <algorithm>
#include <cstdlib>

#include "cov_common.cuh"
#include "rcp_internal.cuh"

namespace rcp {

using namespace covk;

namespace {

constexpr int CELL_SHIFT = 11;                       // 2048-bp cells of the L2-resident table
constexpr int BM_SHIFT = 14;                         // 16384-bp blocks of the shared-memory bitmap
constexpr int CELLS_PER_BIG = ((TILE - 1) >> CELL_SHIFT) + 2;
constexpr int CELLS_PER_SMALL = ((SMALL_MAX - 1) >> CELL_SHIFT) + 2;
constexpr int RTPB = 512;                            // threads of the read passes
constexpr uint32_t NONE = 0xffffffffu;

// tile record, first half: what the read passes need
//   x = global coordinate of the first genomic base of the tile
//   y = tlen (bits 0..15) | reverse (bit 16) | class mask (bits 17..19)      (never 0)
// second half: x = region, y = offset of the tile inside the region's output
struct Tiles {
    uint2* a;
    uint2* b;
};

// Cell table: one 16-byte record per 2048-bp cell = the first tile overlapping the cell, inline
// (x, y as in Tiles::a; y == 0: no tile; z = tile id; w = index of the cell's overflow records
// or NONE).  Overflow records have the same layout and end with a y == 0 sentinel.  One 16-byte
// load answers "which tile does this read hit" for almost every read.
struct Cells {
    uint4* rec;          // [n_cell]
    uint4* ovf;
    uint32_t* cnt;       // [n_cell + 1] tiles per cell (counts down to 0 while slots are handed out)
    uint32_t* ovf_n;     // [n_cell + 1] overflow records per cell (0 or cnt incl. the sentinel)
    uint32_t* ovf_ptr;   // [n_cell + 1] exclusive prefix of ovf_n
    uint32_t* bitmap;    // 1 bit per 16384-bp block: some tile overlaps it
};

__global__ void __launch_bounds__(CTA)
bkt_plan_kernel(int64_t R, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
                const int32_t* __restrict__ end, const int8_t* __restrict__ strand,
                const uint32_t* __restrict__ chrom_off, const int64_t* __restrict__ chrom_len,
                int n_chrom, int ignore_strand, int strand_filter, uint32_t* __restrict__ gs_out,
                int32_t* __restrict__ plen, uint8_t* __restrict__ flags,
                int64_t* __restrict__ nbig, int64_t* __restrict__ nsmall,
                unsigned int* __restrict__ err) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= R) return;
    const int st = strand ? (int)strand[r] : 0;
    uint32_t gs;
    int64_t L;
    const bool null = window_geometry(chrom[r], start[r], end[r], n_chrom, chrom_off, chrom_len,
                                      err, &gs, &L);
    const int32_t len = null ? 0 : (int32_t)L;
    gs_out[r] = gs;
    plen[r] = len;
    flags[r] = (uint8_t)((st < 0 ? 1u : 0u) | (class_mask(st, ignore_strand, strand_filter) << 1));
    nbig[r] = len > SMALL_MAX ? ((int64_t)len + TILE - 1) / TILE : 0;
    nsmall[r] = (len > 0 && len <= SMALL_MAX) ? 1 : 0;
}

// last r in [0, R) with off[r] <= t  (off is an exclusive prefix sum with off[R] = total > t)
__device__ __forceinline__ int64_t owner_of(const int64_t* __restrict__ off, int64_t R, int64_t t) {
    int64_t lo = 0, hi = R;              // answer in [lo, hi)
    while (hi - lo > 1) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(off + mid) <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

// One thread per tile: tile record, the count of every cell it overlaps, its bitmap bits.
__global__ void __launch_bounds__(CTA)
bkt_tiles_kernel(int64_t R, int64_t Tb, int64_t Ts, const int64_t* __restrict__ off_big,
                 const int64_t* __restrict__ off_small, const uint32_t* __restrict__ gs,
                 const int32_t* __restrict__ plen, const uint8_t* __restrict__ flags, Tiles tiles,
                 uint32_t* __restrict__ cell_cnt, uint32_t* __restrict__ bitmap) {
    const int64_t t = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (t >= Tb + Ts) return;
    int64_t r;
    uint32_t o_lo, tlen, tstart;
    if (t < Tb) {
        r = owner_of(off_big, R, t);
        const int j = (int)(t - off_big[r]);
        const int L = plen[r];
        const int m = (L + TILE - 1) / TILE;
        const int tile_len = (((L + m - 1) / m) + ROW - 1) / ROW * ROW;
        o_lo = (uint32_t)(j * tile_len);
        tlen = (uint32_t)min(tile_len, L - (int)o_lo);
        // tiles are cut in OUTPUT space: on a '-' region tile j covers the mirrored positions
        const uint32_t q0 = (flags[r] & 1u) ? (uint32_t)L - o_lo - tlen : o_lo;
        tstart = gs[r] + q0;
    } else {
        r = owner_of(off_small, R, t - Tb);
        o_lo = 0;
        tlen = (uint32_t)plen[r];
        tstart = gs[r];
    }
    tiles.a[t] = make_uint2(tstart, tlen | ((uint32_t)flags[r] << 16));
    tiles.b[t] = make_uint2((uint32_t)r, o_lo);
    const uint32_t last = tstart + tlen - 1u;
    for (uint32_t c = tstart >> CELL_SHIFT; c <= (last >> CELL_SHIFT); c++) atomicAdd(cell_cnt + c, 1u);
    for (uint32_t b = tstart >> BM_SHIFT; b <= (last >> BM_SHIFT); b++)
        atomicOr(bitmap + (b >> 5), 1u << (b & 31u));
}

// cells holding two or more tiles keep all but one in overflow records (+ a sentinel)
__global__ void __launch_bounds__(CTA)
bkt_ovf_count_kernel(int64_t n, const uint32_t* __restrict__ cnt, uint32_t* __restrict__ ovf_n) {
    const int64_t c = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (c >= n) return;
    const uint32_t k = cnt[c];
    ovf_n[c] = k >= 2u ? k : 0u;
}

// Fills the cell table.  cnt counts down to zero while the slots are handed out: slot 0 is the
// inline record, slots 1.. go to the overflow run (the holder of slot 1 also writes the sentinel).
__global__ void __launch_bounds__(CTA)
bkt_cells_kernel(int64_t T, Tiles tiles, Cells cells) {
    const int64_t t = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (t >= T) return;
    const uint2 a = tiles.a[t];
    const uint32_t last = a.x + (a.y & 0xffffu) - 1u;
    for (uint32_t c = a.x >> CELL_SHIFT; c <= (last >> CELL_SHIFT); c++) {
        const uint32_t slot = atomicSub(cells.cnt + c, 1u) - 1u;
        const uint32_t p0 = cells.ovf_ptr[c], p1 = cells.ovf_ptr[c + 1];
        if (slot == 0u) {
            cells.rec[c] = make_uint4(a.x, a.y, (uint32_t)t, p1 > p0 ? p0 : NONE);
        } else {
            cells.ovf[p0 + slot - 1u] = make_uint4(a.x, a.y, (uint32_t)t, 0u);
            if (slot == 1u) cells.ovf[p1 - 1u] = make_uint4(0u, 0u, 0u, 0u);
        }
    }
}

// One (read, tile record) test.  A hit is credited in exactly one cell: the one holding the first
// base of the intersection.  On a hit the read is clipped to the tile and packed as one event
// pair (first covered output | one past the last, << 16), mirrored on '-' regions so that the
// tile kernels only ever scan forwards.
template <bool STRANDED>
__device__ __forceinline__ bool record_hit(const uint4 rec, uint32_t c, uint32_t s, uint32_t e1,
                                           unsigned bit, uint32_t* packed) {
    const uint32_t ts = rec.x, tl = rec.y & 0xffffu;
    if (!(ts < e1 && ts + tl > s)) return false;
    const uint32_t is = max(ts, s);
    if ((is >> CELL_SHIFT) != c) return false;
    if (STRANDED && !((rec.y >> (17 + bit)) & 1u)) return false;
    uint32_t lo = is - ts, hi = min(e1, ts + tl) - ts;           // covered [lo, hi)
    if (rec.y & 0x10000u) {                                       // '-' region: mirror
        const uint32_t l2 = tl - hi;
        hi = tl - lo;
        lo = l2;
    }
    *packed = lo | (hi << 16);
    return true;
}

// ---- pass 1: find ---------------------------------------------------------------------------
// Every read -> the tiles it overlaps.  Persistent CTAs keep the block bitmap in shared memory;
// the reads stream in with 16-byte evict-first loads.  The work is irregular (most reads of a
// sparse mask hit nothing, some hit several tiles), so each warp runs it through two small
// shared-memory queues and stays converged:
//   item queue   (read, cell) pairs that passed the bitmap; a ROUND pops 32 of them, one per
//                lane, loads the 16-byte cell record (or overflow record) and tests it; a record
//                with a successor re-queues the read for the next record
//   hit buffer   (tile, event pair) of the hits; flushed 128+ at a time to the global hit list
//                with ONE atomic reservation and coalesced 8-byte stores
// Each hit also bumps its tile's counter (fire-and-forget RED).  If the hit list overflows its
// capacity the counters are still exact and the caller falls back to bkt_rescatter_kernel.
constexpr int RWARPS = RTPB / 32;
constexpr int QCAP = 64;
constexpr int HB_FLUSH = 128;
constexpr int HB_CAP = HB_FLUSH + 32;
constexpr size_t FIND_SMEM_FIXED = (size_t)RWARPS * (QCAP * sizeof(uint4) + HB_CAP * sizeof(uint2));

struct FindOut {
    uint32_t* tile_cnt;             // 32-bit: the total number of hits is checked to be < 2^32
    uint2* hits;                    // (tile, event pair)
    unsigned long long cap;         // entries available in `hits`
    unsigned long long* hit_n;      // entries reserved so far (> cap: the list is incomplete)
};

template <bool STRANDED>
__global__ void __launch_bounds__(RTPB)
bkt_find_kernel(int64_t n, const uint32_t* __restrict__ g_start,
                const uint32_t* __restrict__ g_end1, const int8_t* __restrict__ strand,
                const uint32_t* __restrict__ bitmap, int bm_words,
                const uint4* __restrict__ cell_rec, const uint4* __restrict__ ovf, FindOut out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint4* q = reinterpret_cast<uint4*>(smem_raw) + (threadIdx.x >> 5) * QCAP;
    uint2* hb = reinterpret_cast<uint2*>(reinterpret_cast<uint4*>(smem_raw) + RWARPS * QCAP) +
                (threadIdx.x >> 5) * HB_CAP;
    uint32_t* bm = reinterpret_cast<uint32_t*>(smem_raw + FIND_SMEM_FIXED);
    for (int i = threadIdx.x; i < bm_words; i += RTPB) bm[i] = bitmap[i];
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    int qn = 0, hn = 0;             // warp-uniform fill levels

    auto flush = [&]() {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(out.hit_n, (unsigned long long)hn);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base + (unsigned long long)hn <= out.cap)
            for (int i = lane; i < hn; i += 32) out.hits[base + i] = hb[i];
        hn = 0;
        __syncwarp();
    };
    // pop the last `cnt` items (cnt <= 32), one per lane
    auto round = [&](int cnt) {
        __syncwarp();
        const bool act = (int)lane < cnt;
        uint4 it = make_uint4(0, 0, 0, 0);
        if (act) it = q[qn - cnt + (int)lane];
        qn -= cnt;
        __syncwarp();
        bool hit = false, more = false;
        uint32_t tile = 0, packed = 0, next = 0;
        if (act) {
            const uint32_t c = it.z & 0x3fffffu;
            const bool is_ovf = (it.w >> 31) != 0u;
            const uint32_t idx = it.w & 0x7fffffffu;
            const uint4 rec = is_ovf ? __ldg(ovf + idx) : __ldg(cell_rec + c);
            if (rec.y != 0u) {
                hit = record_hit<STRANDED>(rec, c, it.x, it.y, it.z >> 30, &packed);
                tile = rec.z;
                if (is_ovf) {
                    more = true;            // the run ends with a y == 0 sentinel
                    next = idx + 1u;
                } else if (rec.w != NONE) {
                    more = true;
                    next = rec.w;
                }
            }
        }
        const unsigned mm = __ballot_sync(0xffffffffu, more);
        if (more) q[qn + __popc(mm & lt)] = make_uint4(it.x, it.y, it.z, 0x80000000u | next);
        qn += __popc(mm);
        const unsigned hm = __ballot_sync(0xffffffffu, hit);
        if (hit) {
            atomicAdd(out.tile_cnt + tile, 1u);
            hb[hn + __popc(hm & lt)] = make_uint2(tile, packed);
        }
        hn += __popc(hm);
        if (hn >= HB_FLUSH) flush();
    };
    // one read per lane (invalid lanes pass e1 = 0)
    auto slot = [&](uint32_t s, uint32_t e1, int st) {
        bool cand = e1 > s;
        const uint32_t c0 = s >> CELL_SHIFT;
        uint32_t c1 = c0;
        if (cand) {
            const uint32_t b0 = s >> BM_SHIFT, b1 = (e1 - 1u) >> BM_SHIFT;
            uint32_t w = bm[b0 >> 5] >> (b0 & 31u);
            if (b1 != b0) w |= bm[b1 >> 5] >> (b1 & 31u);          // rare: one load for most reads
            cand = (b1 > b0 + 1u) || (w & 1u);
            c1 = (e1 - 1u) >> CELL_SHIFT;
        }
        const uint32_t tag = (st > 0 ? 0u : (st < 0 ? 1u : 2u)) << 30;
        // first cell of every candidate, last cell of those that touch two, then (reads longer
        // than a cell: rare) the cells in between
        const unsigned m1 = __ballot_sync(0xffffffffu, cand);
        if (m1 == 0u) return;
        if (cand) q[qn + __popc(m1 & lt)] = make_uint4(s, e1, c0 | tag, 0u);
        qn += __popc(m1);
        while (qn >= 32) round(32);     // a round may re-queue up to 32 items: keep qn < 32
        const bool two = cand && c1 != c0;
        const unsigned m2 = __ballot_sync(0xffffffffu, two);
        if (m2 == 0u) return;
        if (two) q[qn + __popc(m2 & lt)] = make_uint4(s, e1, c1 | tag, 0u);
        qn += __popc(m2);
        while (qn >= 32) round(32);     // a round may re-queue up to 32 items: keep qn < 32
        for (uint32_t cur = c0 + 1u;; cur++) {
            const bool has = two && cur < c1;
            const unsigned m = __ballot_sync(0xffffffffu, has);
            if (m == 0u) break;
            if (has) q[qn + __popc(m & lt)] = make_uint4(s, e1, cur | tag, 0u);
            qn += __popc(m);
            while (qn >= 32) round(32);
        }
    };

    const int64_t n_vec = n >> 2;
    const int64_t warps_total = (int64_t)gridDim.x * RWARPS;
    const int64_t gw = (int64_t)blockIdx.x * RWARPS + (threadIdx.x >> 5);
    for (int64_t base = gw * 32; base < n_vec; base += warps_total * 32) {
        const int64_t v = base + lane;
        uint4 s4 = make_uint4(0, 0, 0, 0), e4 = make_uint4(0, 0, 0, 0);
        char4 t4 = make_char4(0, 0, 0, 0);
        if (v < n_vec) {
            s4 = __ldcs(reinterpret_cast<const uint4*>(g_start) + v);
            e4 = __ldcs(reinterpret_cast<const uint4*>(g_end1) + v);
            if (STRANDED && strand) t4 = __ldcs(reinterpret_cast<const char4*>(strand) + v);
        }
        slot(s4.x, e4.x, t4.x);
        slot(s4.y, e4.y, t4.y);
        slot(s4.z, e4.z, t4.z);
        slot(s4.w, e4.w, t4.w);
    }
    if (gw == 0) {                  // the n % 4 tail
        const int64_t i = n_vec * 4 + lane;
        const bool ok = i < n;
        slot(ok ? g_start[i] : 0u, ok ? g_end1[i] : 0u, (ok && STRANDED && strand) ? (int)strand[i] : 0);
    }
    while (qn > 0) round(min(qn, 32));
    if (hn > 0) flush();
}

// ---- pass 2: place --------------------------------------------------------------------------
// hit list -> per-tile buckets.  `cursor` starts at the tile's bucket offset.
__global__ void __launch_bounds__(CTA)
bkt_place_kernel(unsigned long long n_hits, const uint2* __restrict__ hits,
                 uint32_t* __restrict__ cursor, uint32_t* __restrict__ bucket) {
    // four hits per thread and trip: four independent load -> ATOM -> store chains in flight
    const unsigned long long stride = (unsigned long long)gridDim.x * CTA;
    const unsigned long long n4 = n_hits >> 2;
    for (unsigned long long v = (unsigned long long)blockIdx.x * CTA + threadIdx.x; v < n4; v += stride) {
        const uint4 a = __ldcs(reinterpret_cast<const uint4*>(hits) + 2 * v);
        const uint4 b = __ldcs(reinterpret_cast<const uint4*>(hits) + 2 * v + 1);
        const uint32_t s0 = atomicAdd(cursor + a.x, 1u);
        const uint32_t s1 = atomicAdd(cursor + a.z, 1u);
        const uint32_t s2 = atomicAdd(cursor + b.x, 1u);
        const uint32_t s3 = atomicAdd(cursor + b.z, 1u);
        bucket[s0] = a.y;
        bucket[s1] = a.w;
        bucket[s2] = b.y;
        bucket[s3] = b.w;
    }
    for (unsigned long long i = n4 * 4 + (unsigned long long)blockIdx.x * CTA + threadIdx.x; i < n_hits;
         i += stride) {
        const uint2 h = __ldcs(hits + i);
        bucket[atomicAdd(cursor + h.x, 1u)] = h.y;
    }
}

// ---- pass 2, fallback: the hit list did not fit, walk the reads again -------------------------
template <bool STRANDED>
__device__ __forceinline__ void rescatter_read(uint32_t s, uint32_t e1, int st,
                                               const uint32_t* __restrict__ bm,
                                               const uint4* __restrict__ cell_rec,
                                               const uint4* __restrict__ ovf,
                                               uint32_t* __restrict__ cursor,
                                               uint32_t* __restrict__ bucket) {
    if (e1 <= s) return;
    const uint32_t b0 = s >> BM_SHIFT, b1 = (e1 - 1u) >> BM_SHIFT;
    if (!((b1 > b0 + 1u) || (((bm[b0 >> 5] >> (b0 & 31u)) | (bm[b1 >> 5] >> (b1 & 31u))) & 1u))) return;
    const unsigned bit = st > 0 ? 0u : (st < 0 ? 1u : 2u);
    const uint32_t c1 = (e1 - 1u) >> CELL_SHIFT;
    for (uint32_t c = s >> CELL_SHIFT; c <= c1; c++) {
        uint4 rec = __ldg(cell_rec + c);
        if (rec.y == 0u) continue;
        uint32_t p = rec.w, packed;
        for (;;) {
            if (record_hit<STRANDED>(rec, c, s, e1, bit, &packed))
                bucket[atomicAdd(cursor + rec.z, 1u)] = packed;
            if (p == NONE) break;
            rec = __ldg(ovf + p++);
            if (rec.y == 0u) break;
        }
    }
}

template <bool STRANDED>
__global__ void __launch_bounds__(RTPB)
bkt_rescatter_kernel(int64_t n, const uint32_t* __restrict__ g_start,
                     const uint32_t* __restrict__ g_end1, const int8_t* __restrict__ strand,
                     const uint32_t* __restrict__ bitmap, int bm_words,
                     const uint4* __restrict__ cell_rec, const uint4* __restrict__ ovf,
                     uint32_t* __restrict__ cursor, uint32_t* __restrict__ bucket) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* bm = reinterpret_cast<uint32_t*>(smem_raw);
    for (int i = threadIdx.x; i < bm_words; i += RTPB) bm[i] = bitmap[i];
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * RTPB;
    for (int64_t i = (int64_t)blockIdx.x * RTPB + threadIdx.x; i < n; i += stride)
        rescatter_read<STRANDED>(__ldcs(g_start + i), __ldcs(g_end1 + i),
                                 (STRANDED && strand) ? (int)strand[i] : 0, bm, cell_rec, ovf,
                                 cursor, bucket);
}

// NULL rule (coverage.R:198,224-225): no overlapping read in any tile of the region.
__global__ void __launch_bounds__(CTA)
bkt_null_kernel(int64_t R, int64_t Tb, const int64_t* __restrict__ off_big,
                const int64_t* __restrict__ off_small, const int32_t* __restrict__ plen,
                const uint32_t* __restrict__ tile_cnt, int32_t* __restrict__ len,
                uint8_t* __restrict__ is_null, int64_t* __restrict__ padded,
                unsigned long long* __restrict__ stats /* [0] n_null, [1] total_len */) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (r < R) {
        const int32_t L = plen[r];
        uint32_t hits = 0;          // only zero / non-zero matters
        if (L > SMALL_MAX) {
            for (int64_t t = off_big[r]; t < off_big[r + 1]; t++) hits |= tile_cnt[t];
        } else if (L > 0) {
            hits = tile_cnt[Tb + off_small[r]];
        }
        const bool null = hits == 0;
        const int32_t out = null ? 0 : L;
        len[r] = out;
        is_null[r] = null ? 1 : 0;
        padded[r] = ((int64_t)out + PAD - 1) / PAD * PAD;
        my_null = null ? 1 : 0;
        my_len = (unsigned long long)out;
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

// Everything a tile kernel needs, in one 32-byte record (one dependent load instead of five).
struct __align__(16) TileDesc {
    int64_t out;         // offset of the tile's first output in the dense coverage
    uint32_t b0;         // first bucket entry
    uint32_t n;          // bucket entries
    int32_t tlen;        // outputs; 0 = the region is NULL, nothing to write
    int32_t pad[3];
};

__global__ void __launch_bounds__(CTA)
bkt_desc_kernel(int64_t T, Tiles tiles, const uint32_t* __restrict__ boff,
                const uint8_t* __restrict__ is_null, const int64_t* __restrict__ off,
                TileDesc* __restrict__ desc) {
    const int64_t t = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (t >= T) return;
    const uint2 b = tiles.b[t];
    TileDesc d;
    d.out = off[b.x] + b.y;
    d.b0 = boff[t];
    d.n = boff[t + 1] - boff[t];
    d.tlen = is_null[b.x] ? 0 : (int32_t)(tiles.a[t].y & 0xffffu);
    d.pad[0] = d.pad[1] = d.pad[2] = 0;
    desc[t] = d;
}

__device__ __forceinline__ TileDesc load_desc(const TileDesc* __restrict__ p) {
    const int4 a = __ldg(reinterpret_cast<const int4*>(p));
    const int4 b = __ldg(reinterpret_cast<const int4*>(p) + 1);
    TileDesc d;
    d.out = (int64_t)(((uint64_t)(uint32_t)a.y << 32) | (uint32_t)a.x);
    d.b0 = (uint32_t)a.z;
    d.n = (uint32_t)a.w;
    d.tlen = b.x;
    d.pad[0] = d.pad[1] = d.pad[2] = 0;
    return d;
}

// One tile, RPW rows per warp: zero the shared-memory difference array, add the bucket's event
// pairs with shared-memory atomics, scan, store.  e0 / e1 are the bucket entries this thread
// prefetched (NONE = none).
template <int RPW>
__device__ __forceinline__ void tile_body(int* diff, int* wtot, int tlen, uint32_t n,
                                          const uint32_t* __restrict__ entries, uint32_t e0,
                                          uint32_t e1, int32_t* __restrict__ dst) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int k = 0; k < RPW; k++)       // WARPS * RPW rows = RPW int4 per thread
        reinterpret_cast<int4*>(diff)[k * CTA + tid] = make_int4(0, 0, 0, 0);
    __syncthreads();
    auto add = [&](uint32_t e) {
        const int lo = (int)(e & 0xffffu), hi = (int)(e >> 16);
        atomicAdd(diff + lo, 1);
        if (hi < tlen) atomicSub(diff + hi, 1);
    };
    if (e0 != NONE) add(e0);
    if (e1 != NONE) add(e1);
    for (uint32_t i = 2 * CTA + tid; i < n; i += CTA) add(__ldcs(entries + i));
    __syncthreads();
    block_scan_store_fwd<RPW, true>(diff, tlen, wtot, dst);
}

// Long regions: persistent CTAs walk the tiles.  Nothing the current tile needs is loaded in
// its own iteration: the descriptor is fetched two tiles ahead and the first bucket entries one
// tile ahead, so their latency hides behind the scan and the stores of the tiles in between.
__global__ void __launch_bounds__(CTA, 5)
bkt_tile_kernel(int64_t Tb, const TileDesc* __restrict__ desc, const uint32_t* __restrict__ bucket,
                int32_t* __restrict__ cov) {
    __shared__ __align__(16) int diff[TILE];
    __shared__ int wtot[WARPS];
    const uint32_t tid = threadIdx.x;
    const int64_t step = gridDim.x;
    int64_t t = blockIdx.x;
    if (t >= Tb) return;
    TileDesc none;
    none.out = 0;
    none.b0 = 0;
    none.n = 0;
    none.tlen = 0;
    none.pad[0] = none.pad[1] = 0;
    TileDesc d = load_desc(desc + t);
    TileDesc dn = (t + step < Tb) ? load_desc(desc + t + step) : none;
    uint32_t e0 = NONE, e1 = NONE;                  // NONE never is a valid pair (lo < hi)
    if (tid < d.n) e0 = __ldcs(bucket + d.b0 + tid);
    if (tid + CTA < d.n) e1 = __ldcs(bucket + d.b0 + tid + CTA);
    for (;;) {
        // issue the loads of the following tiles first: dn is already in registers
        const TileDesc dnn = (t + 2 * step < Tb) ? load_desc(desc + t + 2 * step) : none;
        uint32_t f0 = NONE, f1 = NONE;
        if (tid < dn.n) f0 = __ldcs(bucket + dn.b0 + tid);
        if (tid + CTA < dn.n) f1 = __ldcs(bucket + dn.b0 + tid + CTA);
        if (d.tlen > 0) {
            const int rpw = ((d.tlen + ROW - 1) / ROW + WARPS - 1) / WARPS;
            const uint32_t* entries = bucket + d.b0;
            int32_t* dst = cov + d.out;
            switch (rpw) {
                case 1: tile_body<1>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                case 2: tile_body<2>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                case 3: tile_body<3>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                case 4: tile_body<4>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                case 5: tile_body<5>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                case 6: tile_body<6>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
                default: tile_body<7>(diff, wtot, d.tlen, d.n, entries, e0, e1, dst); break;
            }
        }
        t += step;
        if ((tid & 31u) == 0) tma_store_wait_read();    // this warp's bulk store has read `diff`
        if (t >= Tb) break;
        __syncthreads();            // diff and wtot are reused
        d = dn;
        dn = dnn;
        e0 = f0;
        e1 = f1;
    }
}

// Short regions (<= SMALL_MAX bases): one warp per region, warp-private tile, __syncwarp only.
__global__ void __launch_bounds__(CTA)
bkt_small_kernel(int64_t Ts, const TileDesc* __restrict__ desc, const uint32_t* __restrict__ bucket,
                 int32_t* __restrict__ cov) {
    __shared__ __align__(16) int sm[WARPS][SMALL_MAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ts = (int64_t)blockIdx.x * WARPS + warp;
    if (ts >= Ts) return;
    const TileDesc d = load_desc(desc + ts);
    const int L = d.tlen;
    if (L == 0) return;
    int* diff = sm[warp];
    const int nrows = (L + ROW - 1) / ROW;
    for (int i = lane; i < nrows * (ROW / 4); i += 32)
        reinterpret_cast<int4*>(diff)[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    for (uint32_t i = lane; i < d.n; i += 32) {
        const uint32_t e = __ldcs(bucket + d.b0 + i);
        const int lo = (int)(e & 0xffffu), hi = (int)(e >> 16);
        atomicAdd(diff + lo, 1);
        if (hi < L) atomicSub(diff + hi, 1);
    }
    __syncwarp();
    // row by row (a lane-serial scan of 8 rows would put every lane's run in the same banks)
    int32_t* dst = cov + d.out;
    int pre = 0;
    for (int row = 0; row < nrows; row++)
        pre += warp_row_scan_store(diff + row * ROW, pre, 0, false, L - row * ROW, dst + row * ROW);
}

inline unsigned reads_grid(int64_t n, size_t smem) {
    int64_t b = ((n + 3) / 4 + RTPB - 1) / RTPB;
    // persistent CTAs: as many as fit per SM beside their queues and bitmap copies
    int per_sm = 2048 / RTPB;
    while (per_sm > 1 && (size_t)per_sm * (smem + 1024) > 220u * 1024u) per_sm--;
    const int64_t cap = (int64_t)g_ctx.sm_count * per_sm;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

// Device scratch of one call.  Three arenas (one allocation each: the host is on the critical
// path right after the two synchronisation points, and ~30 stream-ordered allocations plus as
// many frees cost more than the small kernels between them): A sized by the regions, B by the
// tiles / cells / reads, C by the hits.  (Arena: rcp_internal.cuh)
struct Work {
    Arena A, B, C;
    uint32_t* gs = nullptr;
    int32_t* plen = nullptr;
    uint8_t* flags = nullptr;
    int64_t* nbig = nullptr;
    int64_t* nsmall = nullptr;
    int64_t* off_big = nullptr;
    int64_t* off_small = nullptr;
    int64_t* padded = nullptr;
    unsigned int* err = nullptr;
    unsigned long long* stats = nullptr;
    Tiles tiles = {nullptr, nullptr};
    Cells cells = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int bm_words = 0;
    uint32_t* tile_cnt = nullptr;             // counts, then (pass 2) bucket cursors
    uint2* hits = nullptr;
    unsigned long long* hit_n = nullptr;
    uint32_t* boff = nullptr;
    uint32_t* bucket = nullptr;
    TileDesc* desc = nullptr;
};

template <bool STRANDED>
int launch_find(const ReadsIdx& rd, const Work& w, unsigned long long cap) {
    const size_t smem = FIND_SMEM_FIXED + (size_t)w.bm_words * 4;
    auto kern = bkt_find_kernel<STRANDED>;
    RCP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FindOut out;
    out.tile_cnt = w.tile_cnt;
    out.hits = w.hits;
    out.cap = cap;
    out.hit_n = w.hit_n;
    kern<<<reads_grid(rd.n, smem), RTPB, smem, g_ctx.stream>>>(
        rd.n, rd.g_start, rd.g_end1, rd.d_strand, w.cells.bitmap, w.bm_words, w.cells.rec,
        w.cells.ovf, out);
    RCP_LAUNCHED();
    return RCP_OK;
}

template <bool STRANDED>
int launch_rescatter(const ReadsIdx& rd, const Work& w) {
    const size_t smem = (size_t)w.bm_words * 4;
    auto kern = bkt_rescatter_kernel<STRANDED>;
    RCP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = (rd.n + RTPB - 1) / RTPB;
    kern<<<(unsigned)std::min<int64_t>(blocks, (int64_t)g_ctx.sm_count * 4), RTPB, smem,
           g_ctx.stream>>>(rd.n, rd.g_start, rd.g_end1, rd.d_strand, w.cells.bitmap, w.bm_words,
                           w.cells.rec, w.cells.ovf, w.tile_cnt, w.bucket);
    RCP_LAUNCHED();
    return RCP_OK;
}

}  // namespace

// may_switch: under RCP_PATH_AUTO the call gives up right after the plan (RCP_SWITCH_TO_INDEX) when
// the mask is dense AND the read set is very large: there the random accesses of the two read
// passes leave L2 (C5 at full size: 200 M reads, 10^6 windows: 12.3 ms against 10.6 ms through
// the sorted index), while for sparse masks or fewer reads the buckets win (C2, C3, C5 / 4).
int coverage_ranges_bucketed(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                             const int32_t* end, const int8_t* strand, int ignore_strand,
                             int strand_filter, int mem, bool may_switch, Coverage* cv) {
    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_chrom.init(chrom, (size_t)R, mem));
    RCP_TRY(d_start.init(start, (size_t)R, mem));
    RCP_TRY(d_end.init(end, (size_t)R, mem));
    RCP_TRY(d_strand.init(strand, (size_t)R, mem));
    // the class test is needed only when some rule can exclude a read (reads without a strand
    // array are all '*': a '+' / '-' filter then keeps nothing)
    const bool stranded = !((strand_filter == RCP_STRAND_ANY) && (ignore_strand || strand == nullptr));

    cv->n_regions = R;
    RCP_TRY(dalloc(&cv->off, (size_t)R + 1));
    RCP_TRY(dalloc(&cv->len, (size_t)R));
    RCP_TRY(dalloc(&cv->is_null, (size_t)R));
    Work w;
    {
        const size_t r = (size_t)R;
        RCP_TRY(w.A.reserve(Arena::pad(r * 4) * 2 + Arena::pad(r) + Arena::pad(r * 8) * 3 +
                            Arena::pad((r + 1) * 8) * 2 + Arena::pad(4) + Arena::pad(24)));
        w.err = w.A.take<unsigned int>(1);            // err and stats first: one memset clears both
        w.stats = w.A.take<unsigned long long>(3);
        w.gs = w.A.take<uint32_t>(r);
        w.plen = w.A.take<int32_t>(r);
        w.flags = w.A.take<uint8_t>(r);
        w.nbig = w.A.take<int64_t>(r);
        w.nsmall = w.A.take<int64_t>(r);
        w.padded = w.A.take<int64_t>(r);
        w.off_big = w.A.take<int64_t>(r + 1);
        w.off_small = w.A.take<int64_t>(r + 1);
        if (w.A.used > w.A.cap) return fail(RCP_ERR_CUDA, "internal: region arena overrun");
    }
    RCP_CUDA(cudaMemsetAsync(w.err, 0, 512, g_ctx.stream));       // err (256 B slot) + stats

    struct Host {
        int64_t Tb, Ts, total_padded, hits;
        unsigned long long stats[3], listed;
        unsigned int err;
    } h = {0, 0, 0, 0, {0, 0, 0}, 0, 0};

    // ---- 1. plan: windows and tile counts ------------------------------------------------
    {
        StageTimer t(ST_BKT_PLAN);
        if (R > 0) {
            bkt_plan_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(
                R, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr, rd.d_chrom_off,
                rd.d_chrom_len, rd.n_chrom, ignore_strand, strand_filter, w.gs, w.plen, w.flags,
                w.nbig, w.nsmall, w.err);
            RCP_LAUNCHED();
        }
        RCP_TRY(exclusive_scan2_i64(w.nbig, w.off_big, w.off_big + R, w.nsmall, w.off_small,
                                    w.off_small + R, R));
    }
    {
        const FetchItem items[3] = {{w.off_big + R, &h.Tb, 8}, {w.off_small + R, &h.Ts, 8}, {w.err, &h.err, 4}};
        RCP_TRY(fetch_and_sync(items, 3));
    }
    if (h.err & 1u) return fail(RCP_ERR_DATA, "a region has a chromosome id outside [0, n_chrom)");
    if (h.err & 2u) return fail(RCP_ERR_DATA, "a region has end < start - 1");
    const int64_t Tb = h.Tb, Ts = h.Ts, T = Tb + Ts;
    if (T > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 coverage tiles");
    int64_t switch_reads = 120000000;
    if (const char* e = getenv("RCP_BKT_SWITCH_READS")) switch_reads = strtoll(e, nullptr, 10);   // tests
    if (may_switch && rd.n >= switch_reads &&
        (double)Tb * TILE + (double)Ts * SMALL_MAX >= 0.25 * (double)rd.chrom_off[(size_t)rd.n_chrom])
        return RCP_SWITCH_TO_INDEX;

    // ---- 2. tiles, cell table, block bitmap -------------------------------------------------
    const int64_t span = (int64_t)rd.chrom_off[(size_t)rd.n_chrom];
    const int64_t n_cell = (span >> CELL_SHIFT) + 2;
    const int64_t pairs = Tb * CELLS_PER_BIG + Ts * CELLS_PER_SMALL;      // (tile, cell) bound
    w.bm_words = (int)(((span >> BM_SHIFT) + 32) / 32);
    // The hit list holds one entry per read by default: enough unless regions overlap heavily
    // (then pass 2 walks the reads again instead).  RCP_BKT_HIT_CAP overrides it (tests).
    unsigned long long hit_cap = (unsigned long long)std::max<int64_t>(rd.n, 4096);
    if (const char* e = getenv("RCP_BKT_HIT_CAP")) hit_cap = strtoull(e, nullptr, 10);
    size_t zero_bytes = 0;
    {
        const size_t t = (size_t)T, c = (size_t)n_cell, ovf_cap = (size_t)(pairs + pairs / 2 + 1);
        RCP_TRY(w.B.reserve(Arena::pad(c * 16) + Arena::pad((c + 1) * 4) * 3 + Arena::pad((size_t)w.bm_words * 4) +
                            Arena::pad((t + 1) * 4) * 2 + Arena::pad(16) + Arena::pad(t * 8) * 2 +
                            Arena::pad(ovf_cap * 16) + Arena::pad((size_t)hit_cap * 8)));
        // zero-initialised block first (ONE memset): cell records, cell counts, bitmap, tile counters,
        // hit counter
        w.cells.rec = w.B.take<uint4>(c);
        w.cells.cnt = w.B.take<uint32_t>(c + 1);
        w.cells.bitmap = w.B.take<uint32_t>((size_t)w.bm_words);
        w.tile_cnt = w.B.take<uint32_t>(t + 1);
        w.hit_n = w.B.take<unsigned long long>(2);
        zero_bytes = w.B.used;
        w.cells.ovf_n = w.B.take<uint32_t>(c + 1);
        w.cells.ovf_ptr = w.B.take<uint32_t>(c + 1);
        w.boff = w.B.take<uint32_t>(t + 1);
        w.tiles.a = w.B.take<uint2>(t);
        w.tiles.b = w.B.take<uint2>(t);
        w.cells.ovf = w.B.take<uint4>(ovf_cap);
        w.hits = w.B.take<uint2>((size_t)hit_cap);
        if (w.B.used > w.B.cap) return fail(RCP_ERR_CUDA, "internal: tile arena overrun");
    }
    {
        StageTimer t(ST_BKT_PLAN);
        RCP_CUDA(cudaMemsetAsync(w.B.base, 0, zero_bytes, g_ctx.stream));
        if (T > 0) {
            bkt_tiles_kernel<<<blocks_for(T, CTA), CTA, 0, g_ctx.stream>>>(
                R, Tb, Ts, w.off_big, w.off_small, w.gs, w.plen, w.flags, w.tiles, w.cells.cnt,
                w.cells.bitmap);
            RCP_LAUNCHED();
            bkt_ovf_count_kernel<<<blocks_for(n_cell + 1, CTA), CTA, 0, g_ctx.stream>>>(
                n_cell + 1, w.cells.cnt, w.cells.ovf_n);
            RCP_LAUNCHED();
            RCP_TRY(exclusive_scan_u32(w.cells.ovf_n, w.cells.ovf_ptr, n_cell + 1, nullptr));
            bkt_cells_kernel<<<blocks_for(T, CTA), CTA, 0, g_ctx.stream>>>(T, w.tiles, w.cells);
            RCP_LAUNCHED();
        }
    }
    // ---- 3. pass 1: find the (read, tile) hits; count them per tile -------------------------
    if (T > 0 && rd.n > 0) {
        StageTimer t(ST_BKT_COUNT);
        RCP_TRY(stranded ? launch_find<true>(rd, w, hit_cap) : launch_find<false>(rd, w, hit_cap));
    }
    // ---- 4. NULL rule, offsets ---------------------------------------------------------------
    {
        StageTimer t(ST_BKT_PLAN);
        if (R > 0) {
            bkt_null_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(
                R, Tb, w.off_big, w.off_small, w.plen, w.tile_cnt, cv->len, cv->is_null, w.padded,
                w.stats);
            RCP_LAUNCHED();
        }
        RCP_TRY(exclusive_scan_i64(w.padded, cv->off, R, cv->off + R));
        RCP_TRY(exclusive_scan_u32(w.tile_cnt, w.boff, T, w.boff + T));
    }
    {
        const FetchItem items[3] = {{cv->off + R, &h.total_padded, 8}, {w.stats, h.stats, 24}, {w.hit_n, &h.listed, 8}};
        RCP_TRY(fetch_and_sync(items, 3));
    }
    cv->path = RCP_PATH_BUCKETS;
    cv->total_padded = h.total_padded;
    cv->n_null = (int64_t)h.stats[0];
    cv->total_len = (int64_t)h.stats[1];
    cv->max_len = (int32_t)h.stats[2];
    RCP_TRY(dalloc(&cv->cov, (size_t)h.total_padded));
    // the find pass counted every hit exactly (64-bit); the per-tile counters and offsets are 32-bit
    if (h.listed > 0xfffffff0ull)
        return fail(RCP_ERR_UNSUPPORTED,
                    "more than 2^32 (read, tile) overlaps: use RCP_PATH_INDEX for this mask");
    h.hits = (int64_t)h.listed;
    if (h.hits == 0) return RCP_OK;                 // every region is NULL
    RCP_TRY(w.C.reserve(Arena::pad((size_t)h.hits * 4) + Arena::pad((size_t)T * sizeof(TileDesc))));
    w.bucket = w.C.take<uint32_t>((size_t)h.hits);
    w.desc = w.C.take<TileDesc>((size_t)T);
    // ---- 5. pass 2: hits -> buckets (the counters become cursors starting at the offsets) -----
    {
        StageTimer t(ST_BKT_SCATTER);
        RCP_CUDA(cudaMemcpyAsync(w.tile_cnt, w.boff, (size_t)T * 4, cudaMemcpyDeviceToDevice,
                                 g_ctx.stream));
        if (h.listed <= hit_cap) {
            const int64_t blocks = ((int64_t)h.listed / 4 + CTA - 1) / CTA + 1;
            bkt_place_kernel<<<(unsigned)std::min<int64_t>(blocks, (int64_t)g_ctx.sm_count * 16), CTA,
                               0, g_ctx.stream>>>(h.listed, w.hits, w.tile_cnt, w.bucket);
            RCP_LAUNCHED();
        } else {
            RCP_TRY(stranded ? launch_rescatter<true>(rd, w) : launch_rescatter<false>(rd, w));
        }
        bkt_desc_kernel<<<blocks_for(T, CTA), CTA, 0, g_ctx.stream>>>(T, w.tiles, w.boff, cv->is_null,
                                                                    cv->off, w.desc);
        RCP_LAUNCHED();
    }
    // ---- 6. tiles -> coverage ---------------------------------------------------------------
    if (Tb > 0) {
        StageTimer t(ST_BKT_TILE);
        int per_sm = 0;     // persistent CTAs: exactly one resident wave
        RCP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bkt_tile_kernel, CTA, 0));
        if (per_sm < 1) per_sm = 1;
        bkt_tile_kernel<<<(unsigned)std::min<int64_t>(Tb, (int64_t)g_ctx.sm_count * per_sm), CTA, 0,
                          g_ctx.stream>>>(Tb, w.desc, w.bucket, cv->cov);
        RCP_LAUNCHED();
    }
    if (Ts > 0) {
        StageTimer t(ST_BKT_SMALL);
        bkt_small_kernel<<<blocks_for(Ts, WARPS), CTA, 0, g_ctx.stream>>>(Ts, w.desc + Tb, w.bucket,
                                                                         cv->cov);
        RCP_LAUNCHED();
    }
    return RCP_OK;
}

}  // namespace rcp
