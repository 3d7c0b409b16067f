// SPLIT path (sm_100a): calcCoverage / coverageFromRanges of the reference
// (/root/reference/R/coverage.R:126-226) straight from the UNSORTED reads, with ONE streaming pass
// over the reads and no per-read random access outside shared memory.
//
//   plan     regions -> windows (geometry / NULL rules of coverage.R:209,217-222), tile counts,
//            storage offsets, and a 1-bit-per-16-kb BLOCK BITMAP of the mask.
//   split    the genome is cut into <= 1024 GROUPS of 2^P positions (P from the genome length
//            alone).  Every read is tested against the bitmap in shared memory; a survivor is
//            packed into ONE 32-bit word (position inside its group | strand class | width) and
//            appended to its group's 32-entry ring in shared memory (one shared-memory atomic).
//            Full 16-entry chunks leave as 64-byte stores into a chunk pool; a chunk carries its
//            group in a 2-byte tag.  No histogram pass, no global atomic per read, no prefix sum
//            over the reads.
//   sort     the chunk tags are counting-sorted by group (one cooperative launch over ~N/16 tags);
//            then one CTA per group sorts the group's candidates by 1-kb sub-bin (shared-memory
//            histogram + cursors) into one dense candidate array and writes the sub-bin offsets.
//   tiles    one WARP per tile (<= 896 outputs of one region): the candidates of the sub-bins
//            under it (reaching back by the widest read) are clipped into a warp-private
//            difference array in shared memory (atomics), scanned, and written as int32 coverage
//            by one TMA bulk store.  No block-wide barrier.
//   NULL     a region none of whose tiles saw a read is NULL (coverage.R:198,224-225).  Its
//            storage is allocated up front (offsets do not depend on the reads), so the host
//            synchronises ONCE per call, right after the plan, and never in the read passes.
//
// HBM traffic: 8-9 B per read once, 4 B per candidate written and read twice (second time from
// L2), 4 B per covered base written once.
#include <algorithm>
#include <cstdlib>
#include <chrono>
#include <cstdio>

#include <type_traits>
#include <vector>

#include <cooperative_groups.h>

#include "cov_common.cuh"
#include "r_rng.cuh"
#include "rcp_internal.cuh"

namespace rcp {

using namespace covk;

namespace {

constexpr int BLK_SHIFT = 14;                         // 16384-bp blocks of the bitmap
#ifndef RCP_SUB_SHIFT
#define RCP_SUB_SHIFT 10
#endif
constexpr int SUB_SHIFT = RCP_SUB_SHIFT;              // sub-bins of the candidate sort (2^SUB_SHIFT bp)
constexpr int NG = 1024;                              // groups (at most)
constexpr int RING = 32;                              // ring entries per group (power of two)
constexpr int CH = 16;                                // entries per chunk (64 bytes)
#ifndef RCP_SPLIT_ST
#define RCP_SPLIT_ST 1024
#endif
constexpr int ST = RCP_SPLIT_ST;                      // threads of the split kernel
constexpr int ROUND_VEC = 2048;                       // 16-byte vectors (of 4 reads) per CTA round
constexpr int VPT = ROUND_VEC / ST;                   // vectors per thread and round
constexpr int SLAB = 64;                              // chunks a warp takes from the pool at a time
// position bits of a candidate word: split_position_bits (rcp_internal.cuh), 16..22, for NG groups
static_assert(NG == 1024, "split_position_bits assumes at most 1024 groups");
constexpr int GT = 1024;                              // threads of the group kernel
constexpr int CS = 1024;                              // threads of the chunk-sort kernels
constexpr int WT = 7 * ROW;                           // outputs of a warp tile (896); regions <= 1024 bp are ONE tile
constexpr int WT_ONE = SMALL_MAX;
static_assert(NG % ST == 0 && ROUND_VEC % ST == 0, "the flush phase maps thread t to the groups t, t + ST, ...");
static_assert(RING == 2 * CH, "a ring holds two chunks");
static_assert(SLAB >= 64, "one flush phase of a warp needs up to 64 chunks");

// Block table: one 32-bit word per 16 blocks.  Bit k (k < 16): block 16 w + k is in the mask;
// bit 16 + k: the block AFTER it is (so that one load also answers for a read that crosses into
// the next block).
__device__ __forceinline__ void sp_mark_block(uint32_t* __restrict__ tab, uint32_t b) {
    atomicOr(tab + (b >> 4), 1u << (b & 15u));
    if (b > 0) atomicOr(tab + ((b - 1u) >> 4), 0x10000u << ((b - 1u) & 15u));
}

// ---------------------------------------------------------------------------------- plan ------
__global__ void __launch_bounds__(CTA)
sp_plan_kernel(int64_t R, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
               const int32_t* __restrict__ end, const int8_t* __restrict__ strand,
               const uint32_t* __restrict__ chrom_off, const int64_t* __restrict__ chrom_len,
               int n_chrom, int ignore_strand, int strand_filter, uint32_t* __restrict__ gs_out,
               int32_t* __restrict__ plen, uint8_t* __restrict__ flags, int64_t* __restrict__ ntile,
               int64_t* __restrict__ padded, uint32_t* __restrict__ tab, unsigned int* __restrict__ err,
               unsigned long long* __restrict__ pstats /* [0] total len [1] max len [2] 2^32 - min len */,
               unsigned long long* __restrict__ zero5 /* the coverage's stats words: cleared here */) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r < 5) zero5[r] = 0ull;
    unsigned long long my_len = 0;
    if (r < R) {
        const int st = strand ? (int)strand[r] : 0;
        uint32_t gs;
        int64_t L;
        const bool null = window_geometry(chrom[r], start[r], end[r], n_chrom, chrom_off, chrom_len,
                                          err, &gs, &L);
        const int32_t len = null ? 0 : (int32_t)L;
        gs_out[r] = gs;
        plen[r] = len;
        flags[r] = (uint8_t)((st < 0 ? 1u : 0u) | (class_mask(st, ignore_strand, strand_filter) << 1));
        ntile[r] = len > WT_ONE ? ((int64_t)len + WT - 1) / WT : (len > 0 ? 1 : 0);
        padded[r] = ((int64_t)len + PAD - 1) / PAD * PAD;
        my_len = (unsigned long long)len;
        if (len > 0) {
            const uint32_t b1 = (gs + (uint32_t)len - 1u) >> BLK_SHIFT;
            for (uint32_t b = gs >> BLK_SHIFT; b <= b1; b++) sp_mark_block(tab, b);
        }
    }
    unsigned long long my_max = my_len, my_inv = my_len ? 0x100000000ull - my_len : 0ull;
    for (int d = 16; d > 0; d >>= 1) {
        my_len += __shfl_xor_sync(0xffffffffu, my_len, d);
        my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
        my_inv = max(my_inv, __shfl_xor_sync(0xffffffffu, my_inv, d));
    }
    if ((threadIdx.x & 31) == 0 && my_len) {
        atomicAdd(&pstats[0], my_len);
        atomicMax(&pstats[1], my_max);
        atomicMax(&pstats[2], my_inv);
    }
}

__device__ __forceinline__ int64_t sp_owner_of(const int64_t* __restrict__ off, int64_t R, int64_t t) {
    int64_t lo = 0, hi = R;
    while (hi - lo > 1) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(off + mid) <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

// Everything a tile kernel needs in one 32-byte record.
struct __align__(16) SpDesc {
    int64_t out;         // offset of the tile's first output in the dense coverage
    uint32_t c0;         // first candidate
    uint32_t n;          // candidates to look at
    int32_t tlen;        // outputs
    uint32_t cts;        // tile start in compacted coordinates, low P bits
    uint32_t flags;      // bit0 reverse, bits1..3 strand classes the region counts
    uint32_t region;
};

// One thread per tile: where it lies (tiles are cut in OUTPUT space, as in the other paths: on a
// '-' region tile j covers the mirrored positions) and which candidates can reach it: those that
// start from (tile start - widest read + 1) on: the run of the sub-bins [first, last] in boff (the
// group sort is queued before this kernel: the host learns the tile count while it runs).
// bound (nullptr: fused or int32 storage): the most reads any tile applies -- n words plus the long
// reads -- goes to this word, one atomicMax per warp.  Each read adds at most 1 to a position, so
// no count of the call exceeds it.
__global__ void __launch_bounds__(CTA)
sp_tiles_kernel(int64_t R, int64_t T, const int64_t* __restrict__ off_tile, const uint32_t* __restrict__ gs,
                const int32_t* __restrict__ plen, const uint8_t* __restrict__ flags,
                const int64_t* __restrict__ cov_off /* nullptr: fused, `out` = offset inside the region
                                                       | first bin the tile meets << 32 */,
                const int32_t* __restrict__ edge, int n_bins,
                uint32_t max_w, uint32_t pmask, const uint32_t* __restrict__ boff, SpDesc* __restrict__ desc,
                uint32_t* __restrict__ tabs,
                const uint32_t* __restrict__ lxs, const uint32_t* __restrict__ lmax, uint32_t ln,
                uint2* __restrict__ lrange, unsigned long long* __restrict__ bound) {
    const int64_t t = (int64_t)blockIdx.x * CTA + threadIdx.x;
    const unsigned live = __ballot_sync(0xffffffffu, t < T);      // the low lanes of the warp
    if (t >= T) return;
    const int64_t r = sp_owner_of(off_tile, R, t);
    const int L = plen[r];
    uint32_t o_lo = 0, tlen = (uint32_t)L;
    if (L > WT_ONE) {
        o_lo = (uint32_t)(t - off_tile[r]) * WT;
        tlen = (uint32_t)min(WT, L - (int)o_lo);
    }
    const uint32_t q0 = (flags[r] & 1u) ? (uint32_t)L - o_lo - tlen : o_lo;
    const uint32_t tstart = gs[r] + q0;
    const uint32_t first = tstart >= max_w ? tstart - max_w + 1u : 0u;
    SpDesc d;
    d.out = cov_off ? cov_off[r] + o_lo : (int64_t)o_lo;
    if (!cov_off) {                         // last bin with edge <= o_lo
        int a = 0, b = n_bins;
        while (b - a > 1) {
            const int mid = (a + b) >> 1;
            if (__ldg(edge + mid) <= (int)o_lo) a = mid;
            else b = mid;
        }
        d.out |= (int64_t)a << 32;
    }
    d.c0 = __ldg(boff + (first >> SUB_SHIFT));
    d.n = __ldg(boff + ((tstart + tlen - 1u) >> SUB_SHIFT) + 1u) - d.c0;
    d.tlen = (int32_t)tlen;
    d.cts = tstart & pmask;
    d.flags = flags[r];
    d.region = (uint32_t)r;
    desc[t] = d;
    uint32_t most = d.n;
    if (ln) {           // the handle keeps long reads aside: those that can meet this tile
        tabs[t] = tstart;
        const uint32_t hi = tstart + tlen - 1u;
        uint32_t a = 0, b = ln;
        while (a < b) {
            const uint32_t mid = a + ((b - a) >> 1);
            if (__ldg(lxs + mid) < hi + 1u) a = mid + 1;
            else b = mid;
        }
        const uint32_t c1 = a;
        a = 0;
        b = c1;
        while (a < b) {
            const uint32_t mid = a + ((b - a) >> 1);
            if (__ldg(lmax + mid) < tstart + 1u) a = mid + 1;
            else b = mid;
        }
        lrange[t] = make_uint2(a, c1);
        most = most + (c1 - a) < most ? 0xffffffffu : most + (c1 - a);
    }
    if (bound) {
        most = __reduce_max_sync(live, most);
        if ((threadIdx.x & 31) == 0) atomicMax(bound, (unsigned long long)most);
    }
}

// --------------------------------------------------------------------------------- split ------
// shared-memory accesses by 32-bit shared address (no generic-pointer arithmetic in the hot loop)
__device__ __forceinline__ uint2 lds64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ int lds_s8(uint32_t a) {
    int v;
    asm volatile("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts8(uint32_t a, int v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atoms_add(uint32_t a, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}

struct SplitOut {
    uint32_t* pool;          // chunks of CH entries
    uint16_t* meta;          // per chunk: group << 5 | entries (0: unused slot)
    uint32_t* pool_next;     // chunks handed out so far (in SLABs); [1]: rounds handed out so far
};

// Shared memory of the split kernel: rings | ring counters | block table.
constexpr size_t sp_split_smem(int words) {
    return (size_t)NG * RING * 4 + (size_t)NG * 4 + (size_t)words * 4;
}
constexpr size_t SP_SMEM_MAX = 232448;                // 227 KB: the most one CTA can have on sm_100

// A round = ST x RPT reads.  Per read: one table load answers "is any block it touches in the
// mask"; a survivor takes a slot of its group's ring with ONE shared-memory atomic and stores its
// packed word there.  Then the CTA meets, thread t flushes the complete chunks of ring t, and reads
// that found their ring full go round again.  A warp that has seen a full ring (coordinate-sorted
// input: everything goes to one group) sends whole 16-entry runs of one group straight to a pool
// chunk from then on.
template <bool STRANDED>
__global__ void __launch_bounds__(ST, 1)
sp_split_kernel(int64_t n, const uint32_t* __restrict__ g_start, const uint32_t* __restrict__ g_end1,
                const int8_t* __restrict__ strand, const uint32_t* __restrict__ tab_g, int words, int P,
                uint32_t max_pack_w, SplitOut out) {
    extern __shared__ __align__(16) unsigned char sp_smem[];
    const int tid = threadIdx.x;
    const unsigned lane = tid & 31, lt = (1u << lane) - 1u;
    const uint32_t ring_a = (uint32_t)__cvta_generic_to_shared(sp_smem);     // NG * RING words
    const uint32_t cnt_a = ring_a + NG * RING * 4;                            // NG: ring start << 16 | fill
    const uint32_t tab_a = cnt_a + NG * 4;                                    // block table
    for (int i = tid; i < words; i += ST) sts32(tab_a + i * 4, tab_g[i]);
    for (int i = tid; i < NG; i += ST) sts32(cnt_a + i * 4, 0u);
    __syncthreads();
    const uint32_t pmask = (1u << P) - 1u;
    const int wsh = STRANDED ? P + 2 : P;
    uint32_t slab_next = 0, slab_end = 0;          // this warp's share of the chunk pool
    uint32_t spare = 0;                            // lane 0: the next slab, requested ahead of need
    bool have_spare = false;
    bool hot = false;                              // this warp has met a full ring

    // `total` chunks for this warp (warp-uniform); chunk i of them is chunk_at(i)
    uint32_t a_rem = 0, a_old = 0, a_new = 0;
    auto alloc = [&](uint32_t total) {
        a_rem = slab_end - slab_next;
        a_old = slab_next;
        a_new = 0;
        if (total > a_rem) {
            if (!have_spare && lane == 0) spare = atomicAdd(out.pool_next, (uint32_t)SLAB);
            a_new = __shfl_sync(0xffffffffu, spare, 0);
            have_spare = false;
            slab_next = a_new + (total - a_rem);
            slab_end = a_new + SLAB;
        } else {
            slab_next += total;
        }
        // request the next slab well before this one runs out: the atomic's round trip then
        // overlaps the following rounds instead of stalling the whole CTA at a barrier
        if (!have_spare && slab_end - slab_next < (uint32_t)SLAB / 2) {
            if (lane == 0) spare = atomicAdd(out.pool_next, (uint32_t)SLAB);
            have_spare = true;
        }
    };
    auto chunk_at = [&](uint32_t i) { return i < a_rem ? a_old + i : a_new + (i - a_rem); };

    // thread t owns the groups t, t + ST, ... here: every complete chunk of a ring leaves as one
    // 64-byte store
    auto flush_phase = [&](bool final_pass) {
#pragma unroll 1
        for (int grp = tid; grp < NG; grp += ST) {
            const uint32_t w = lds32(cnt_a + grp * 4);
            const uint32_t raw = w & 0xffffu, start = w >> 16;
            const uint32_t nn = min(raw, (uint32_t)RING);
            const uint32_t k = final_pass ? (nn > 0u ? 1u : 0u) : nn / CH;
            const unsigned m1 = __ballot_sync(0xffffffffu, k >= 1u), m2 = __ballot_sync(0xffffffffu, k >= 2u);
            const uint32_t total = __popc(m1) + __popc(m2);
            if (total) {                                // warp-uniform
                const uint32_t idx = __popc(m1 & lt) + __popc(m2 & lt);
                alloc(total);
                for (uint32_t j = 0; j < k; j++) {
                    const uint32_t c = chunk_at(idx + j);
                    const uint32_t src = ring_a + (uint32_t)grp * RING * 4 + (((start + CH * j) & (RING - 1)) << 2);
                    uint4* dst = reinterpret_cast<uint4*>(out.pool + (size_t)c * CH);
                    const uint4 a = lds128(src), b = lds128(src + 16), cc = lds128(src + 32), d = lds128(src + 48);
                    __stcs(dst, a);
                    __stcs(dst + 1, b);
                    __stcs(dst + 2, cc);
                    __stcs(dst + 3, d);
                    out.meta[c] = (uint16_t)(((uint32_t)grp << 5) | (final_pass ? nn : (uint32_t)CH));
                }
            }
            if (k || raw > (uint32_t)RING)
                sts32(cnt_a + grp * 4, final_pass ? 0u : ((((start + CH * k) & (RING - 1)) << 16) | (nn - CH * k)));
        }
    };

    // is any block the read touches in the mask?  (crossing reads look at the "next block" bit)
    auto keep_read = [&](uint32_t s, uint32_t e1) -> bool {
        const uint32_t t = lds32(tab_a + ((s >> (BLK_SHIFT + 2)) & 0xfffffffcu)) >> ((s >> BLK_SHIFT) & 15u);
        const bool cross = ((e1 - 1u) >> BLK_SHIFT) != (s >> BLK_SHIFT);
        return ((t & 1u) | (cross & ((t >> 16) & 1u))) & (e1 - s <= max_pack_w);    // wider: the long-read list
    };
    auto pack = [&](uint32_t s, uint32_t e1, int st) -> uint32_t {
        uint32_t word = (s & pmask) | ((e1 - s) << wsh);
        if (STRANDED) word |= (st > 0 ? 0u : (st < 0 ? 1u : 2u)) << P;
        return word;
    };
    // one insertion attempt; false: the ring is full until the next flush
    auto insert = [&](uint32_t g, uint32_t pk) -> bool {
        const uint32_t old = atoms_add(cnt_a + g * 4, 1u);
        const uint32_t slot = old & 0xffffu;
        if (slot >= (uint32_t)RING) return false;
        sts32(ring_a + g * (RING * 4) + ((((old >> 16) + slot) & (RING - 1)) << 2), pk);
        return true;
    };
    // hot warps: when every pending read of this k is about ONE group, whole 16-entry runs go
    // straight to pool chunks; the rest takes the ring
    auto direct = [&](bool want, uint32_t g, uint32_t pk) -> bool {
        const unsigned mo = __ballot_sync(0xffffffffu, want);
        if (mo == 0u) return want;
        const uint32_t g0 = __shfl_sync(0xffffffffu, g, __ffs(mo) - 1);
        const uint32_t nact = __popc(mo);
        if (nact < (uint32_t)CH || !__all_sync(0xffffffffu, !want || g == g0)) return want;
        const uint32_t nfull = nact / CH;
        alloc(nfull);
        const uint32_t r = __popc(mo & lt);           // rank among the pending lanes
        if (want && r < nfull * CH) {
            const uint32_t c = chunk_at(r / CH);
            out.pool[(size_t)c * CH + (r & (CH - 1))] = pk;
            if ((r & (CH - 1)) == 0) out.meta[c] = (uint16_t)((g0 << 5) | (uint32_t)CH);
            return false;
        }
        return want;
    };

    constexpr int RPT = 4 * VPT;                    // reads per thread and round
    // Reads whose ring was full wait here (thread-local memory: a rare path, so that the common one
    // keeps no per-read registers and the next round's loads can stay in flight).
    uint32_t fg[RPT], fp[RPT];
    uint32_t nf = 0;
    auto take = [&](uint32_t sv, uint32_t ev, int tv) {
        const uint32_t g = sv >> P, pk = pack(sv, ev, tv);
        bool want = keep_read(sv, ev);
        if (hot) want = direct(want, g, pk);
        if (want && !insert(g, pk)) {
            fg[nf] = g;
            fp[nf] = pk;
            nf++;
        }
    };
    // barrier, flush, barrier; then the reads that found their ring full go round again
    auto finish_round = [&]() {
        for (;;) {
            hot = hot || __any_sync(0xffffffffu, nf != 0u);
            const int any = __syncthreads_or(nf != 0u);
            flush_phase(false);
            __syncthreads();
            if (!any) break;
            uint32_t mx = nf;                                   // warp-uniform trip count (direct votes)
            for (int d = 16; d > 0; d >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
            uint32_t kept = 0;
            for (uint32_t i = 0; i < mx; i++) {
                const bool mine = i < nf;
                const uint32_t g = mine ? fg[i] : 0u, pk = mine ? fp[i] : 0u;
                bool want = mine;
                if (hot) want = direct(want, g, pk);
                if (want && !insert(g, pk)) {
                    fg[kept] = g;
                    fp[kept] = pk;
                    kept++;
                }
            }
            nf = kept;
        }
    };

    // round r covers the 16-byte vectors [r * ROUND_VEC, (r + 1) * ROUND_VEC): thread t takes the
    // vectors r * ROUND_VEC + h * ST + t (coalesced across the CTA).  The loads of the NEXT round are
    // issued vector by vector as this round's reads are consumed, and stay in flight through the
    // rest of the insertions, both barriers and the flush.
    // Rounds are handed out by a global counter, not by a fixed stride: when the kernel shares the
    // GPU (the NCCL gather of the previous step holds a few SMs) the CTAs that start late simply
    // take fewer rounds, instead of running a second wave that doubles the kernel's time.  The
    // index of the round after next is fetched by thread 0 during a round and published through
    // shared memory at that round's barriers.
    __shared__ int next_round[2];
    const int64_t n_vec = n >> 2;
    const int rounds = (int)((n_vec + ROUND_VEC - 1) / ROUND_VEC);
    if (tid == 0) {
        next_round[0] = (int)atomicAdd(out.pool_next + 1, 1u);
        next_round[1] = (int)atomicAdd(out.pool_next + 1, 1u);
    }
    __syncthreads();
    int round = next_round[0], nr = next_round[1];
    __syncthreads();
    uint4 s4[VPT], e4[VPT];
    char4 t4[VPT];
    auto load = [&](int rd, int h) {
        const int64_t v = (int64_t)rd * ROUND_VEC + h * ST + tid;
        s4[h] = e4[h] = make_uint4(0, 0, 0, 0);
        t4[h] = make_char4(0, 0, 0, 0);
        if (rd < rounds && v < n_vec) {
            s4[h] = __ldcs(reinterpret_cast<const uint4*>(g_start) + v);
            e4[h] = __ldcs(reinterpret_cast<const uint4*>(g_end1) + v);
            if (STRANDED && strand) t4[h] = __ldcs(reinterpret_cast<const char4*>(strand) + v);
        }
    };
#pragma unroll
    for (int h = 0; h < VPT; h++) load(round, h);
    for (int it = 0; round < rounds; it++) {
        unsigned after = 0;
        if (tid == 0) after = atomicAdd(out.pool_next + 1, 1u);     // in flight during the round
#pragma unroll
        for (int h = 0; h < VPT; h++) {
            take(s4[h].x, e4[h].x, t4[h].x);
            take(s4[h].y, e4[h].y, t4[h].y);
            take(s4[h].z, e4[h].z, t4[h].z);
            take(s4[h].w, e4[h].w, t4[h].w);
            load(nr, h);                    // into the registers just consumed
        }
        if (tid == 0) next_round[it & 1] = (int)min(after, 0x7fffffffu);
        finish_round();                     // (its barriers publish next_round[it & 1])
        round = nr;
        nr = next_round[it & 1];
    }
    if (blockIdx.x == 0) {              // the n % 4 tail
        const int64_t i = n_vec * 4 + tid;
        const bool in = i < n;
        const uint32_t sv = in ? g_start[i] : 0u, ev = in ? g_end1[i] : 0u;
        take(sv, ev, (in && STRANDED && strand) ? (int)strand[i] : 0);
        finish_round();
    }
    flush_phase(true);                   // what is left in the rings: one partial chunk per group
}

// ---------------------------------------------------------------------- chunks by group -------
// Counting sort of the chunk tags: per-CTA histograms over a contiguous range of pool slots, a
// column-wise prefix, then the placement with shared-memory cursors.
__device__ __forceinline__ void sp_slot_range(uint32_t n_slots, uint32_t* lo, uint32_t* hi) {
    const uint32_t per = ((n_slots + gridDim.x - 1) / gridDim.x + CS - 1) / CS * CS;
    *lo = min(n_slots, blockIdx.x * per);
    *hi = min(n_slots, *lo + per);
}

// One cooperative launch (64 CTAs, all resident): histogram of this CTA's slot range, grid barrier,
// every CTA works out its own cursors from the whole count table (64 x 1024 words from L2: cheaper
// than a second barrier around a one-CTA prefix), placement.  CTA 0 also writes cb[g] = first
// chunk-list entry of group g (cb[NG] = chunks in all).
__global__ void __launch_bounds__(CS)
sp_chunk_lists_kernel(const uint16_t* __restrict__ meta, const uint32_t* __restrict__ pool_next,
                      uint32_t* __restrict__ col /* [gridDim.x][NG] */, uint32_t* __restrict__ cb,
                      uint32_t* __restrict__ list /* slot << 5 | entries */) {
    static_assert(CS == NG, "thread g of a CTA owns group g");
    __shared__ uint32_t h[NG];
    __shared__ uint32_t wsum[NG / 32];
    const int g = threadIdx.x;
    h[g] = 0;
    __syncthreads();
    uint32_t lo, hi;
    sp_slot_range(*pool_next, &lo, &hi);
    for (uint32_t i = lo + threadIdx.x; i < hi; i += CS) {
        const uint32_t m = meta[i];
        if (m & 31u) atomicAdd(&h[m >> 5], 1u);
    }
    __syncthreads();
    col[(size_t)blockIdx.x * NG + g] = h[g];
    cooperative_groups::this_grid().sync();
    uint32_t tot = 0, before = 0;
    for (unsigned c = 0; c < gridDim.x; c++) {
        const uint32_t v = __ldcg(col + (size_t)c * NG + g);
        tot += v;
        if (c < blockIdx.x) before += v;
    }
    uint32_t inc = tot;
    const unsigned lane = g & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (unsigned)d) inc += o;
    }
    if (lane == 31) wsum[g >> 5] = inc;
    __syncthreads();
    uint32_t run = inc - tot;
    for (int k = 0; k < (g >> 5); k++) run += wsum[k];
    if (blockIdx.x == 0) {
        cb[g] = run;
        if (g == NG - 1) cb[NG] = run + tot;
    }
    h[g] = run + before;                // cursor of this CTA for group g
    __syncthreads();
    for (uint32_t i = lo + threadIdx.x; i < hi; i += CS) {
        const uint32_t m = meta[i];
        if (m & 31u) list[atomicAdd(&h[m >> 5], 1u)] = (i << 5) | (m & 31u);
    }
}

// ------------------------------------------------------------------- candidates by sub-bin -----
// One CTA per group (2^P positions of the genome): histogram of the group's candidates over its
// 1-kb sub-bins, prefix, placement.  The sorted group is assembled in SHARED MEMORY (cursors are
// shared-memory atomics) and leaves with coalesced 16-byte stores: a 4-byte store per candidate
// to a random place costs as much as a global atomic (~180 G/s for the whole chip).  A group too
// large for shared memory scatters directly.  The group's output starts at CH * cb[g] (its chunk
// capacity: the partial chunks leave a hole of zero words -- width 0, never a hit -- at the end
// of the group's range).
constexpr size_t GSMEM = 220 * 1024;      // dynamic shared memory of the group kernel (1 CTA per SM)

__global__ void __launch_bounds__(GT, 1)
sp_group_kernel(const uint32_t* __restrict__ pool, const uint32_t* __restrict__ list,
                const uint32_t* __restrict__ cb, int n_groups, int nb /* sub-bins of a group */,
                uint32_t pmask, uint32_t* __restrict__ cand, uint32_t* __restrict__ boff) {
    extern __shared__ __align__(16) uint32_t gsm[];
    uint32_t* h = gsm;                             // nb counts, then cursors
    uint32_t* out = gsm + nb;                      // the sorted group
    const uint32_t cap = (uint32_t)(GSMEM / 4) - (uint32_t)nb;
    __shared__ uint32_t wsum[GT / 32];
    const int tid = threadIdx.x, g = blockIdx.x;
    for (int i = tid; i < nb; i += GT) h[i] = 0;
    __syncthreads();
    const uint32_t c0 = cb[g], c1 = cb[g + 1];
    // four lanes per chunk (16 bytes each): a warp reads 8 chunks with one 16-byte load per lane
    const uint32_t q4 = (tid & 3) * 4, cw = tid >> 2;
    constexpr uint32_t CPS = GT / 4, U = 4;                       // chunks per CTA step, steps in flight
    // list entries are fetched one iteration ahead of the chunks they name
    auto stream = [&](auto&& use) {
        uint32_t le[U], ln[U];
        uint4 e[U];
#pragma unroll
        for (uint32_t u = 0; u < U; u++) {
            const uint32_t i = c0 + cw + u * CPS;
            ln[u] = i < c1 ? __ldg(list + i) : 0u;
        }
        for (uint32_t i0 = c0 + cw; i0 < c1; i0 += CPS * U) {
#pragma unroll
            for (uint32_t u = 0; u < U; u++) {
                le[u] = ln[u];
                e[u] = make_uint4(0u, 0u, 0u, 0u);
                if (q4 < (le[u] & 31u))
                    e[u] = __ldg(reinterpret_cast<const uint4*>(pool + (size_t)(le[u] >> 5) * CH + q4));
            }
#pragma unroll
            for (uint32_t u = 0; u < U; u++) {
                const uint32_t i = i0 + CPS * U + u * CPS;
                ln[u] = i < c1 ? __ldg(list + i) : 0u;
            }
#pragma unroll
            for (uint32_t u = 0; u < U; u++) {
                const uint32_t f = le[u] & 31u;
                use(e[u], q4 < f, q4 + 1 < f, q4 + 2 < f, q4 + 3 < f);
            }
        }
    };
    auto sub = [&](uint32_t e) { return (e & pmask) >> SUB_SHIFT; };
    stream([&](uint4 e, bool v0, bool v1, bool v2, bool v3) {
        if (v0) atomicAdd(&h[sub(e.x)], 1u);
        if (v1) atomicAdd(&h[sub(e.y)], 1u);
        if (v2) atomicAdd(&h[sub(e.z)], 1u);
        if (v3) atomicAdd(&h[sub(e.w)], 1u);
    });
    // placement: the four cursor atomics of a 16-byte word are issued back to back and the four
    // stores follow, so that a thread waits for ONE shared-memory round trip per word, not four
    auto place = [&](uint32_t* dst) {
        stream([&](uint4 e, bool v0, bool v1, bool v2, bool v3) {
            uint32_t p0 = 0, p1 = 0, p2 = 0, p3 = 0;
            if (v0) p0 = atomicAdd(&h[sub(e.x)], 1u);
            if (v1) p1 = atomicAdd(&h[sub(e.y)], 1u);
            if (v2) p2 = atomicAdd(&h[sub(e.z)], 1u);
            if (v3) p3 = atomicAdd(&h[sub(e.w)], 1u);
            if (v0) dst[p0] = e.x;
            if (v1) dst[p1] = e.y;
            if (v2) dst[p2] = e.z;
            if (v3) dst[p3] = e.w;
        });
    };
    __syncthreads();
    // exclusive prefix of the nb counts: warp w owns the bins [w * pw, (w + 1) * pw) and walks them
    // 32 at a time (consecutive lanes, consecutive bins: no bank conflicts); the warp bases follow
    // from the warp totals
    constexpr int NW = GT / 32;
    const int pw = (nb + NW - 1) / NW;
    const unsigned lane = tid & 31;
    const int wb0 = (tid >> 5) * pw, wb1 = min(nb, wb0 + pw);
    uint32_t carry = 0;
    for (int b = wb0 + (int)lane; b - (int)lane < wb1; b += 32) {
        const uint32_t c = b < wb1 ? h[b] : 0u;
        uint32_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= (unsigned)d) inc += o;
        }
        if (b < wb1) h[b] = carry + inc - c;                    // relative to the warp's first bin
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) wsum[tid >> 5] = carry;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
    for (int k = 0; k < NW; k++) {
        if (k < (tid >> 5)) wbase += wsum[k];
        total += wsum[k];
    }
    const uint32_t base = c0 * CH;
    for (int b = wb0 + (int)lane; b < wb1; b += 32) {
        const uint32_t o = h[b] + wbase;
        h[b] = o;                                               // cursor
        boff[(size_t)g * nb + b] = base + o;
    }
    if (g == n_groups - 1 && tid == 0) boff[(size_t)n_groups * nb] = base + total;
    __syncthreads();
    if (total > cap) {          // a huge group: plain scatter, then the hole.  (Sorting it in slices of
                                // sub-bins that fit shared memory was tried: every slice is one more
                                // pass over the group's chunks, C4 1.32 -> 1.74 ms.)
        place(cand + base);
        for (uint32_t i = base + total + tid; i < c1 * CH; i += GT) cand[i] = 0u;
        return;
    }
    place(out);
    // zero words up to the group's chunk capacity (a multiple of CH, so of 4): the hole
    const uint32_t full = (c1 - c0) * CH;
    for (uint32_t i = total + tid; i < min(full, (total + 3u) & ~3u); i += GT) out[i] = 0u;
    __syncthreads();
    const uint32_t n4 = (total + 3u) >> 2;                       // 16-byte words holding candidates
    uint4* dst = reinterpret_cast<uint4*>(cand + base);           // base is a multiple of CH words
    for (uint32_t i = tid; i < n4; i += GT) dst[i] = reinterpret_cast<const uint4*>(out)[i];
    for (uint32_t i = n4 * 4 + tid; i < full; i += GT) cand[base + i] = 0u;
}

// ------------------------------------------------------------------------ long reads ----------
// Reads wider than the packed word allows stay out of the binned index: start-sorted, with the
// running maximum of their ends, they are looked up per tile (GRanges masks) or per element
// (GRangesList masks) and applied whole.
struct LongIdx {
    uint32_t n;
    const uint32_t* xs;      // sorted starts
    const uint32_t* e1;      // end + 1
    const int8_t* st;        // strand (nullptr: '*')
    const uint32_t* maxe1;   // running max of e1
};

// CTA c owns LONG_PER consecutive reads: it counts its long reads, reserves their places with ONE
// global atomic, and writes them (the second look at the reads comes from L1 / L2).  The total is
// known beforehand (the map kernel counts them), the order is settled by the sort that follows.
constexpr int LONG_PER = CTA * 16;
__global__ void __launch_bounds__(CTA)
sp_long_collect_kernel(int64_t n, const uint32_t* __restrict__ s, const uint32_t* __restrict__ e1,
                       uint32_t max_pack_w, unsigned int* __restrict__ cursor_g, uint32_t cap,
                       uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    __shared__ unsigned cnt, cursor;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    const int64_t lo = (int64_t)blockIdx.x * LONG_PER, hi = min(n, lo + LONG_PER);
    unsigned c = 0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += CTA) c += (e1[i] - s[i] > max_pack_w) && (e1[i] > s[i]);
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if (lane == 0 && c) atomicAdd(&cnt, c);
    __syncthreads();
    if (cnt == 0) return;                                   // (uniform: read after the barrier)
    if (threadIdx.x == 0) cursor = atomicAdd(cursor_g, cnt);
    __syncthreads();
    for (int64_t b0 = lo + (threadIdx.x & ~31u); b0 < hi; b0 += CTA) {        // warp-uniform trip count
        const int64_t i = b0 + lane;
        const bool is = i < hi && e1[i] - s[i] > max_pack_w && e1[i] > s[i];
        const unsigned m = __ballot_sync(0xffffffffu, is);
        if (m == 0u) continue;
        unsigned k = 0;
        if (lane == 0) k = atomicAdd(&cursor, (unsigned)__popc(m));        // shared memory
        k = __shfl_sync(0xffffffffu, k, 0) + __popc(m & ((1u << lane) - 1u));
        if (is && k < cap) {
            keys[k] = s[i];
            idx[k] = (uint32_t)i;
        }
    }
}

__global__ void __launch_bounds__(CTA)
sp_long_gather_kernel(uint32_t n, const uint32_t* __restrict__ idx, const uint32_t* __restrict__ e1,
                      const int8_t* __restrict__ st, uint32_t* __restrict__ o_e1, int8_t* __restrict__ o_st) {
    const uint32_t i = blockIdx.x * CTA + threadIdx.x;
    if (i >= n) return;
    o_e1[i] = e1[idx[i]];
    if (st) o_st[i] = st[idx[i]];
}

__device__ __forceinline__ uint32_t sp_lower_bound(const uint32_t* __restrict__ a, uint32_t lo, uint32_t hi, uint32_t v) {
    while (lo < hi) {               // first index with a[i] >= v
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// long reads that can meet [lo, hi] (global, closed): start <= hi and the running max of end + 1 > lo
__device__ __forceinline__ uint2 sp_long_range(const LongIdx& lg, uint32_t lo, uint32_t hi) {
    const uint32_t c1 = sp_lower_bound(lg.xs, 0, lg.n, hi + 1u);
    const uint32_t c0 = sp_lower_bound(lg.maxe1, 0, c1, lo + 1u);
    return make_uint2(c0, c1);
}

// --------------------------------------------------------------------------------- tiles ------
__device__ __forceinline__ SpDesc sp_load_desc(const SpDesc* __restrict__ p) {
    const int4 a = __ldg(reinterpret_cast<const int4*>(p));
    const int4 b = __ldg(reinterpret_cast<const int4*>(p) + 1);
    SpDesc d;
    d.out = (int64_t)(((uint64_t)(uint32_t)a.y << 32) | (uint32_t)a.x);
    d.c0 = (uint32_t)a.z;
    d.n = (uint32_t)a.w;
    d.tlen = b.x;
    d.cts = (uint32_t)b.y;
    d.flags = (uint32_t)b.z;
    d.region = (uint32_t)b.w;
    return d;
}

// One candidate against one tile: adds its two events to the difference array (mirrored on '-'
// regions, so the scan only ever runs forwards).  Returns true on a hit.
template <bool STRANDED>
__device__ __forceinline__ bool sp_apply(uint32_t e, const SpDesc& d, int P, int* diff) {
    const int sh = 32 - P;
    const int rel = ((int)((e - d.cts) << sh)) >> sh;              // candidate start - tile start
    uint32_t w = e >> (STRANDED ? P + 2 : P);
    if (STRANDED && !((d.flags >> (1u + ((e >> P) & 3u))) & 1u)) w = 0;
    int lo = max(rel, 0), hi = min(rel + (int)w, d.tlen);
    if (lo >= hi) return false;
    if (d.flags & 1u) {
        const int l2 = d.tlen - hi;
        hi = d.tlen - lo;
        lo = l2;
    }
    atomicAdd(diff + lo, 1);
    if (hi < d.tlen) atomicSub(diff + hi, 1);
    return true;
}

// The same for the hot loop of the warp-tile kernel: `rev` is a template parameter (the caller
// branches once per tile, warp-uniformly), both events are PREDICATED shared-memory reductions (no
// divergent branch around them), addresses are 32-bit shared addresses.  cls = the region's strand
// classes (flags >> 1).
template <bool STRANDED, bool REV>
__device__ __forceinline__ bool sp_apply_fast(uint32_t e, uint32_t cts, int tlen, uint32_t cls, int P,
                                              uint32_t diff_a) {
    const int sh = 32 - P;
    const int rel = ((int)((e - cts) << sh)) >> sh;                // candidate start - tile start
    int w = (int)(e >> (STRANDED ? P + 2 : P));
    if (STRANDED) w = ((cls >> ((e >> P) & 3u)) & 1u) ? w : 0;
    const int lo = max(rel, 0), hi = min(rel + w, tlen);
    const int a = REV ? tlen - hi : lo;                            // +1 here
    const int b = REV ? tlen - lo : hi;                            // -1 here unless it is the tile's end
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.lt.s32 p, %0, %1;\n\t"
        "setp.lt.and.s32 q, %2, %3, p;\n\t"
        "@p red.shared.add.s32 [%4], 1;\n\t"
        "@q red.shared.add.s32 [%5], -1;\n\t"
        "}" ::"r"(lo), "r"(hi), "r"(b), "r"(tlen), "r"(diff_a + (uint32_t)a * 4u), "r"(diff_a + (uint32_t)b * 4u)
        : "memory");
    return lo < hi;
}

// Lane-serial forward scan of a warp-private tile of RPW rows (RPW * 128 ints, zero-padded): lane
// l owns the RPW * 4 consecutive ints at l * RPW * 4 (16-byte loads with a lane stride of
// RPW * 16 bytes: conflict-free for odd RPW); the lane sums its run, one warp scan orders the
// lanes, the run is rescanned from the right start and written back in place; the TMA unit then
// stores the tile as ONE bulk copy (cp.async.bulk.global.shared::cta), so no thread spends LSU
// wavefronts on the 4 B / base output.  O = uint16_t (narrow storage): the counts are packed into
// the first half of the tile buffer (lane l's 4 * RPW of them at byte l * 8 * RPW) and stored the
// same way; the store runs to the next multiple of 8 counts, inside the region's padding.
template <int RPW, class O = int32_t>
__device__ __forceinline__ void warp_scan_store_fwd(int* diff, int tlen, O* __restrict__ dst) {
    const int lane = threadIdx.x & 31;
    int* mine = diff + lane * 4 * RPW;
    int4 v[RPW];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        v[k] = *(reinterpret_cast<const int4*>(mine) + k);
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
    const int inc = warp_inclusive_scan(sum);
    int run = inc - sum;
    if (sizeof(O) == 2) __syncwarp();       // every lane has read its run before the packed half is written
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        int4 o;
        o.x = (run += v[k].x);
        o.y = (run += v[k].y);
        o.z = (run += v[k].z);
        o.w = (run += v[k].w);
        if (sizeof(O) == 2)
            *(reinterpret_cast<uint2*>(diff) + lane * RPW + k) =
                make_uint2(((uint32_t)o.x & 0xffffu) | ((uint32_t)o.y << 16), ((uint32_t)o.z & 0xffffu) | ((uint32_t)o.w << 16));
        else
            *(reinterpret_cast<int4*>(mine) + k) = o;
    }
    __syncwarp();
    if (lane == 0) {
        fence_proxy_async_smem();
        constexpr int E = 16 / (int)sizeof(O);      // elements per 16-byte granule
        tma_store_1d(dst, diff, (uint32_t)((tlen + E - 1) & ~(E - 1)) * (uint32_t)sizeof(O));
        tma_store_commit();
    }
}

// 8 rows (a whole region of 897..1024 bp) in narrow storage: row by row (conflict-free, like the
// int32 case), each lane storing its 4 counts as one 8-byte word; the region's padding takes the
// ragged tail.
__device__ __forceinline__ void warp_rows_store_u16(const int* diff, int tlen, uint16_t* __restrict__ dst) {
    const int lane = threadIdx.x & 31;
    int pre = 0;
    for (int row = 0; row * ROW < tlen; row++) {
        const int4 v = *(reinterpret_cast<const int4*>(diff + row * ROW) + lane);
        const int i0 = v.x, i1 = i0 + v.y, i2 = i1 + v.z, i3 = i2 + v.w;
        const int inc = warp_inclusive_scan(i3);
        const int ex = pre + inc - i3;
        if (row * ROW + lane * 4 < tlen)
            *reinterpret_cast<uint2*>(dst + row * ROW + lane * 4) =
                make_uint2(((uint32_t)(ex + i0) & 0xffffu) | ((uint32_t)(ex + i1) << 16),
                           ((uint32_t)(ex + i2) & 0xffffu) | ((uint32_t)(ex + i3) << 16));
        pre += __shfl_sync(0xffffffffu, inc, 31);
    }
}

// FUSED coverage -> bins: what a tile hands on instead of its coverage.  The regions have ONE
// common length, so one edge table serves them all (edge[i] = first output of bin i, n + 1
// entries; splitVector's seeded layout, util.R:74-80).  The tile adds, for every bin it meets,
// the sum of its part of the bin to the bin's 64-bit accumulator (a bin may straddle tiles);
// integer sums are exact, so the matrix equals the two-stage path's bit for bit.
struct FusedBins {
    const int32_t* edge;                 // n + 1
    int n;
    int64_t R;
    unsigned long long* acc;             // [n][R]
};

// Scan of a FUSED tile: the lane-serial scan of warp_scan_store_fwd run TWICE in registers, so that
// the tile holds S[k] = c[0] + ... + c[k] (the running sum of the COVERAGE, modulo 2^32) instead of
// the coverage: a bin's part of the tile is then S[hi - 1] - S[lo - 1], two shared-memory loads
// instead of a serial sum of its bases.  Exact as long as the true sum fits 32 bits, which the
// warp checks (coverage below 2^22 everywhere in the tile, <= 1024 bases); otherwise (returns
// false) the tile holds the coverage itself and the bins are summed base by base.
template <int RPW>
__device__ __forceinline__ bool warp_scan_prefix2(int* diff) {
    const int lane = threadIdx.x & 31;
    int* mine = diff + lane * 4 * RPW;
    int4 v[RPW];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        v[k] = *(reinterpret_cast<const int4*>(mine) + k);
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
    const int inc = warp_inclusive_scan(sum);
    const int run0 = inc - sum;
    int run = run0, cmax = 0;
    uint32_t tot = 0;                       // sum of this lane's coverage values
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        run += v[k].x; tot += (uint32_t)run; cmax = max(cmax, run);
        run += v[k].y; tot += (uint32_t)run; cmax = max(cmax, run);
        run += v[k].z; tot += (uint32_t)run; cmax = max(cmax, run);
        run += v[k].w; tot += (uint32_t)run; cmax = max(cmax, run);
    }
    const bool small = __reduce_max_sync(0xffffffffu, cmax) < (1 << 22);
    uint32_t acc = 0;
    if (small) {
        uint32_t incs = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, incs, d);
            if (lane >= d) incs += o;
        }
        acc = incs - tot;
    }
    run = run0;
#pragma unroll
    for (int k = 0; k < RPW; k++) {
        int4 o;
        run += v[k].x; acc += (uint32_t)run; o.x = small ? (int)acc : run;
        run += v[k].y; acc += (uint32_t)run; o.y = small ? (int)acc : run;
        run += v[k].z; acc += (uint32_t)run; o.z = small ? (int)acc : run;
        run += v[k].w; acc += (uint32_t)run; o.w = small ? (int)acc : run;
        *(reinterpret_cast<int4*>(mine) + k) = o;
    }
    __syncwarp();
    return small;
}

// prefixed: the tile holds S (warp_scan_prefix2 returned true), else the coverage
__device__ __forceinline__ void tile_to_bins(const int* tile, const SpDesc& d, const FusedBins& fb, bool prefixed) {
    const int lane = threadIdx.x & 31;
    const int o_lo = (int)(uint32_t)d.out, o_hi = o_lo + d.tlen;
    const int a = (int)(d.out >> 32);    // last bin with edge <= o_lo (sp_tiles_kernel)
    for (int i = a + lane; i < fb.n; i += 32) {
        const int e0 = __ldg(fb.edge + i);
        if (e0 >= o_hi) break;
        const int lo = max(e0, o_lo) - o_lo, hi = min(__ldg(fb.edge + i + 1), o_hi) - o_lo;
        unsigned long long s = 0;
        if (prefixed) {
            if (hi > lo) s = (uint32_t)tile[hi - 1] - (lo > 0 ? (uint32_t)tile[lo - 1] : 0u);
        } else {
            for (int k = lo; k < hi; k++) s += (unsigned long long)(unsigned int)tile[k];
        }
        if (s) atomicAdd(fb.acc + (size_t)i * fb.R + d.region, s);
    }
}

// acc -> the matrix (column-major, like acc): mean of the bin, times the scale; NULL rows are zero
__global__ void __launch_bounds__(CTA)
sp_bins_finish_kernel(FusedBins fb, const int32_t* __restrict__ plen, const uint8_t* __restrict__ region_hit,
                      double scale, double* __restrict__ out, int64_t ld, uint8_t* __restrict__ is_null) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= fb.R) return;
    const int i = blockIdx.y;
    const bool null = plen[r] == 0 || region_hit[r] == 0;
    double v = 0.0;
    if (!null) {
        const int w = __ldg(fb.edge + i + 1) - __ldg(fb.edge + i);
        v = scale * ((double)(long long)fb.acc[(size_t)i * fb.R + r] / (double)w);
    }
    out[(size_t)i * ld + r] = v;
    if (i == 0 && is_null) is_null[r] = null ? 1 : 0;
}

// 16-byte asynchronous copies global -> shared memory (no register staging): the candidates of the
// NEXT tile land in a warp-private buffer while the current tile is built, scanned and stored.
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One WARP per tile (<= 896 outputs; a region <= 1024 bp is one tile): no block-wide barrier
// anywhere.  Persistent warps; descriptors are fetched two tiles ahead, and the first CBUF candidate
// words of the next tile are copied into shared memory (cp.async) during the current tile.  The
// staged range starts at the 16-byte boundary below the tile's first candidate and ends at the one
// above its last.  The extra words belong to neighbouring sub-bins -- possibly of another group, or
// more than 2^(P-1) positions away, where the P-bit distance to the tile wraps and a read far away
// would land inside the tile -- so they are applied as zero words (width 0, never a hit).
// Longer candidate lists continue from global memory, 128 at a time.
#ifndef RCP_WTILE_OCC
#define RCP_WTILE_OCC 4
#endif
constexpr int CBUF = 256;                   // staged candidate words per tile and buffer
constexpr size_t WTILE_SMEM = (size_t)WARPS * (WT_ONE * 4 + 2 * CBUF * 4 + 4 * sizeof(SpDesc));
template <bool STRANDED, bool FUSED>
__global__ void __launch_bounds__(CTA, RCP_WTILE_OCC)
sp_wtile_kernel(int64_t T, const SpDesc* __restrict__ desc, const uint32_t* __restrict__ cand, int P,
                int32_t* __restrict__ cov, uint8_t* __restrict__ region_hit, FusedBins fb, LongIdx lg,
                const uint32_t* __restrict__ tabs, const uint2* __restrict__ lrange,
                const unsigned long long* __restrict__ bound) {
    extern __shared__ __align__(16) unsigned char wt_smem[];
    const bool narrow = !FUSED && cov_narrow(bound);       // the same for every warp of the grid
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;
    int* diff = reinterpret_cast<int*>(wt_smem) + warp * WT_ONE;
    const uint32_t* cs = reinterpret_cast<const uint32_t*>(wt_smem + (size_t)WARPS * WT_ONE * 4) + warp * 2 * CBUF;
    const SpDesc* ring = reinterpret_cast<const SpDesc*>(wt_smem + (size_t)WARPS * (WT_ONE * 4 + 2 * CBUF * 4)) + warp * 4;
    const uint32_t cs_a = (uint32_t)__cvta_generic_to_shared(cs);
    const uint32_t ring_a = (uint32_t)__cvta_generic_to_shared(ring);
    const int64_t step = (int64_t)gridDim.x * WARPS;
    int64_t t = (int64_t)blockIdx.x * WARPS + warp;
    if (t >= T) return;
    // descriptor of this warp's tile number j (tile t0 + j * step) -> ring slot j & 3, by two lanes
    auto stage_desc = [&](int64_t tile, int j) {
        if (lane < 2 && tile < T)
            cp_async16(ring_a + (uint32_t)(j & 3) * (uint32_t)sizeof(SpDesc) + lane * 16u,
                       reinterpret_cast<const int4*>(desc + tile) + lane);
    };
    // the 16-byte units of [c0 & ~3, ...) that hold the first candidates of a tile
    auto stage_cands = [&](uint32_t c0, uint32_t n, int buf) {
        const uint32_t a0 = c0 & ~3u;
        const uint32_t units = min(((c0 - a0) + n + 3u) >> 2, (uint32_t)(CBUF / 4));
#pragma unroll
        for (int k = 0; k < CBUF / 128; k++) {
            const uint32_t u = (uint32_t)k * 32u + lane;
            if (u < units) cp_async16(cs_a + (uint32_t)buf * (CBUF * 4) + u * 16u, cand + a0 + u * 4u);
        }
    };
    stage_desc(t, 0);
    stage_desc(t + step, 1);
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
    stage_cands(ring[0].c0, ring[0].n, 0);
    cp_async_commit();
    int buf = 0;
    constexpr int B = 4;
    // iteration j: the group committed one iteration ago (candidates of tile j, descriptor of tile
    // j + 1) has had a whole tile's time to land; the next group (candidates of j + 1, descriptor
    // of j + 2) is issued before tile j is built
    for (int j = 0;; j++) {
        cp_async_wait<0>();
        __syncwarp();
        const SpDesc d = ring[j & 3];
        const bool more = t + step < T;
        if (more) {
            const SpDesc* nx = ring + ((j + 1) & 3);
            stage_cands(nx->c0, nx->n, buf ^ 1);
        }
        stage_desc(t + 2 * step, j + 2);
        cp_async_commit();
        const int rows = (d.tlen + ROW - 1) / ROW;
        for (int k = 0; k < rows; k++) reinterpret_cast<int4*>(diff)[k * 32 + lane] = make_int4(0, 0, 0, 0);
        __syncwarp();
        bool hit = false;
        const uint32_t a0 = d.c0 & ~3u;
        const uint32_t lead = d.c0 - a0;
        const uint32_t words = lead + d.n;                              // from a0 on
        const uint32_t staged = min((words + 3u) & ~3u, (uint32_t)CBUF);
        const uint32_t mine_a = cs_a + (uint32_t)buf * (CBUF * 4) + lane * 4u;
        const uint32_t diff_a = (uint32_t)__cvta_generic_to_shared(diff);
        const uint32_t cls = d.flags >> 1;
        auto apply_all = [&](auto rev_tag) {
            constexpr bool REV = decltype(rev_tag)::value;
#pragma unroll 4
            for (uint32_t i = lane; i < staged; i += 32) {
                uint32_t e = lds32(mine_a + (i - lane) * 4u);
                if (i < lead || i >= words) e = 0u;                     // outside [c0, c0 + n)
                hit |= sp_apply_fast<STRANDED, REV>(e, d.cts, d.tlen, cls, P, diff_a);
            }
#if defined(RCP_EXP_MODE) && RCP_EXP_MODE == 2     // timing experiment: staged candidates only (wrong results)
            if (d.tlen >= 0) return;
#endif
            for (uint32_t i0 = CBUF; i0 < words; i0 += B * 32) {       // a long list: the rest from global memory
                uint32_t e[B];
#pragma unroll
                for (int k = 0; k < B; k++) {
                    const uint32_t i = i0 + (uint32_t)k * 32u + lane;
                    e[k] = i < words ? __ldg(cand + a0 + i) : 0u;       // 0: width 0, never a hit
                }
#pragma unroll
                for (int k = 0; k < B; k++) hit |= sp_apply_fast<STRANDED, REV>(e[k], d.cts, d.tlen, cls, P, diff_a);
            }
        };
#if defined(RCP_EXP_MODE) && RCP_EXP_MODE == 1     // timing experiment: no candidates applied (wrong results)
        if (d.tlen < 0) apply_all(std::true_type{});
#else
        if (d.flags & 1u) apply_all(std::true_type{});
        else apply_all(std::false_type{});
#endif
        if (lg.n) {             // the reads kept out of the binned index
            const uint2 lr = lrange[t];
            const uint32_t ts = tabs[t];
            for (uint32_t i = lr.x + lane; i < lr.y; i += 32) {
                const uint32_t rs = __ldg(lg.xs + i), re1 = __ldg(lg.e1 + i);
                const int st = lg.st ? (int)__ldg(lg.st + i) : 0;
                const uint32_t cls = st > 0 ? 0u : (st < 0 ? 1u : 2u);
                if (!((d.flags >> (1u + cls)) & 1u)) continue;
                if (rs >= ts + (uint32_t)d.tlen || re1 <= ts) continue;
                int lo = (int)(max(rs, ts) - ts), hi = (int)(min(re1, ts + (uint32_t)d.tlen) - ts);
                if (d.flags & 1u) {
                    const int l2 = d.tlen - hi;
                    hi = d.tlen - lo;
                    lo = l2;
                }
                atomicAdd(diff + lo, 1);
                if (hi < d.tlen) atomicSub(diff + hi, 1);
                hit = true;
            }
        }
        hit = __any_sync(0xffffffffu, hit);
        __syncwarp();
        if (FUSED) {
            if (hit) {                                          // a tile without a read adds nothing
                bool prefixed = false;
                switch (rows) {
                    case 1: prefixed = warp_scan_prefix2<1>(diff); break;
                    case 2: prefixed = warp_scan_prefix2<2>(diff); break;
                    case 3: prefixed = warp_scan_prefix2<3>(diff); break;
                    case 4: prefixed = warp_scan_prefix2<4>(diff); break;
                    case 5: prefixed = warp_scan_prefix2<5>(diff); break;
                    case 6: prefixed = warp_scan_prefix2<6>(diff); break;
                    case 7: prefixed = warp_scan_prefix2<7>(diff); break;
                    default: prefixed = warp_scan_prefix2<8>(diff); break;
                }
                tile_to_bins(diff, d, fb, prefixed);
            }
        } else if (narrow) {
            uint16_t* dst = reinterpret_cast<uint16_t*>(cov) + d.out;
            switch (rows) {
                case 1: warp_scan_store_fwd<1>(diff, d.tlen, dst); break;
                case 2: warp_scan_store_fwd<2>(diff, d.tlen, dst); break;
                case 3: warp_scan_store_fwd<3>(diff, d.tlen, dst); break;
                case 4: warp_scan_store_fwd<4>(diff, d.tlen, dst); break;
                case 5: warp_scan_store_fwd<5>(diff, d.tlen, dst); break;
                case 6: warp_scan_store_fwd<6>(diff, d.tlen, dst); break;
                case 7: warp_scan_store_fwd<7>(diff, d.tlen, dst); break;
                default: warp_rows_store_u16(diff, d.tlen, dst); break;
            }
        } else {
            int32_t* dst = cov + d.out;
            switch (rows) {
                case 1: warp_scan_store_fwd<1>(diff, d.tlen, dst); break;
                case 2: warp_scan_store_fwd<2>(diff, d.tlen, dst); break;
                case 3: warp_scan_store_fwd<3>(diff, d.tlen, dst); break;
                case 4: warp_scan_store_fwd<4>(diff, d.tlen, dst); break;
                case 5: warp_scan_store_fwd<5>(diff, d.tlen, dst); break;
                case 6: warp_scan_store_fwd<6>(diff, d.tlen, dst); break;
                case 7: warp_scan_store_fwd<7>(diff, d.tlen, dst); break;
                default: {      // 8 rows (a whole region of 897..1024 bp): row by row, conflict-free
                    int pre = 0;
                    for (int row = 0; row < rows; row++)
                        pre += warp_row_scan_store(diff + row * ROW, pre, 0, false, d.tlen - row * ROW, dst + row * ROW);
                }
            }
        }
        if (hit && lane == 0) region_hit[d.region] = 1;
        t += step;
        if (!FUSED && lane == 0) tma_store_wait_read();     // the bulk store has read the tile
        if (!more) break;
        __syncwarp();
        buf ^= 1;
    }
}

// ---------------------------------------------------------------------- GRangesList masks -----
// coverageFromRanges on a GRangesList element (coverage.R:177-178,202-207): all ranges (exons) of
// the element stitched into one vector; a read overlapping k ranges of the element counts k times
// on every range it touches (coverage.R:190-192).
struct ListPlan {
    const int64_t* ptr;      // G + 1
    const int8_t* rstrand;   // per range (may be nullptr)
    uint32_t* xgs;           // per range: global start (after the zero-index drop)
    uint32_t* xge;           //            global end; xge + 1 == xgs marks a zero-width range
    int32_t* xoff;           //            offset of the range inside the stitched element
    uint2* lrange;           // per element: the long reads that can meet its span
};

// err bits: 1 chrom id, 2 end < start-1, 4 ranges of one element on different chromosomes
__global__ void __launch_bounds__(CTA)
sp_list_plan_kernel(int64_t G, ListPlan lp, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
                    const int32_t* __restrict__ end, const uint32_t* __restrict__ chrom_off,
                    const int64_t* __restrict__ chrom_len, int n_chrom, int32_t* __restrict__ plen,
                    uint8_t* __restrict__ flags, int64_t* __restrict__ ntile, int64_t* __restrict__ padded,
                    unsigned int* __restrict__ err, unsigned long long* __restrict__ pstats, LongIdx lg) {
    const int64_t g = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_len = 0;
    if (g < G) {
        const int64_t a = lp.ptr[g], b = lp.ptr[g + 1];
        bool null = (b <= a);
        bool simple = true;
        int64_t L = 0;
        int st0 = 0;
        uint32_t lo = 0xffffffffu, hi = 0;
        if (!null) {
            const int c = chrom[a];
            st0 = lp.rstrand ? (int)lp.rstrand[a] : 0;       // strand of the FIRST range (coverage.R:185)
            if (c < 0 || c >= n_chrom) {
                atomicOr(err, 1u);
                null = true;
            } else {
                const int64_t clen = chrom_len[c];
                const uint32_t coff = chrom_off[c];
                int64_t prev_end = -1;
                for (int64_t i = a; i < b; i++) {
                    int64_t s = start[i], e = end[i];
                    // ascending, disjoint, non-empty ranges of one strand: the multiplicity of a read
                    // follows from its neighbours in the list alone (sp_ltile_kernel)
                    if (s <= prev_end || e < s || (lp.rstrand && lp.rstrand[i] != lp.rstrand[a])) simple = false;
                    prev_end = e;
                    if (chrom[i] != c) atomicOr(err, 4u);
                    if (e < s - 1) { atomicOr(err, 2u); null = true; }
                    if (s < 0 || e > clen) null = true;      // coverage.R:206 inside the tryCatch
                    if (s == 0) s = 1;
                    int64_t w = e - s + 1;
                    if (w < 0) w = 0;
                    const uint32_t gs = coff + (uint32_t)(s > 0 ? s : 0);
                    lp.xgs[i] = gs;
                    lp.xge[i] = gs + (uint32_t)w - 1u;
                    lp.xoff[i] = (int32_t)L;
                    L += w;
                    if (w > 0) {
                        lo = min(lo, gs);
                        hi = max(hi, gs + (uint32_t)w - 1u);
                    }
                }
                if (L == 0 || L > 0x7fffffff) null = true;
            }
        }
        const int32_t len = null ? 0 : (int32_t)L;
        lp.lrange[g] = (lg.n && !null) ? sp_long_range(lg, lo, hi) : make_uint2(0u, 0u);
        plen[g] = len;
        flags[g] = (uint8_t)((st0 < 0 ? 1u : 0u) | (simple ? 2u : 0u));
        ntile[g] = len > WT_ONE ? ((int64_t)len + WT - 1) / WT : (len > 0 ? 1 : 0);
        padded[g] = ((int64_t)len + PAD - 1) / PAD * PAD;
        my_len = (unsigned long long)len;
    }
    unsigned long long my_max = my_len;
    for (int d = 16; d > 0; d >>= 1) {
        my_len += __shfl_xor_sync(0xffffffffu, my_len, d);
        my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
    }
    if ((threadIdx.x & 31) == 0 && my_len) {
        atomicAdd(&pstats[0], my_len);
        atomicMax(&pstats[1], my_max);
    }
}

// Number of ranges of the element [a, b) the read [rs, re1) hits under the strand rules
// (coverage.R:190-192).  `simple` elements (ascending, disjoint, one strand): the read is known to
// overlap range q, the other hits are q's neighbours.  Otherwise every range is tested.
__device__ __forceinline__ int sp_multiplicity(const ListPlan& lp, int64_t a, int64_t b, int64_t q, bool simple,
                                               uint32_t rs, uint32_t re1, int rst, int ignore_strand,
                                               int strand_filter) {
    if (simple) {
        if (!strand_ok(rst, lp.rstrand ? (int)__ldg(lp.rstrand + a) : 0, ignore_strand, strand_filter)) return 0;
        int mult = 1;
        for (int64_t z = q + 1; z < b && __ldg(lp.xgs + z) < re1; z++) mult++;
        for (int64_t z = q - 1; z >= a && __ldg(lp.xge + z) >= rs; z--) mult++;
        return mult;
    }
    int mult = 0;
    for (int64_t z = a; z < b; z++) {
        const uint32_t zs = __ldg(lp.xgs + z), ze = __ldg(lp.xge + z);
        if (ze + 1u == zs) continue;
        if (rs <= ze && re1 > zs &&
            strand_ok(rst, lp.rstrand ? (int)__ldg(lp.rstrand + z) : 0, ignore_strand, strand_filter))
            mult++;
    }
    return mult;
}

// tiles of the stitched vectors: `cts` holds the tile's first STITCHED position
__global__ void __launch_bounds__(CTA)
sp_list_tiles_kernel(int64_t G, int64_t T, const int64_t* __restrict__ off_tile, const int32_t* __restrict__ plen,
                     const uint8_t* __restrict__ flags, const int64_t* __restrict__ cov_off,
                     SpDesc* __restrict__ desc) {
    const int64_t t = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (t >= T) return;
    const int64_t g = sp_owner_of(off_tile, G, t);
    const int L = plen[g];
    uint32_t o_lo = 0, tlen = (uint32_t)L;
    if (L > WT_ONE) {
        o_lo = (uint32_t)(t - off_tile[g]) * WT;
        tlen = (uint32_t)min(WT, L - (int)o_lo);
    }
    SpDesc d;
    d.out = cov_off[g] + o_lo;
    d.c0 = d.n = 0;
    d.tlen = (int32_t)tlen;
    d.cts = (flags[g] & 1u) ? (uint32_t)L - o_lo - tlen : o_lo;
    d.flags = flags[g];
    d.region = (uint32_t)g;
    desc[t] = d;
}

// One warp per tile of a stitched vector.  For every range piece under the tile the warp reads the
// candidates of the sub-bins that can reach it; a candidate that overlaps the range adds its
// multiplicity (the number of ranges of the element it hits under the strand rules) on the piece.
template <bool STRANDED>
__global__ void __launch_bounds__(CTA, 4)
sp_ltile_kernel(int64_t T, const SpDesc* __restrict__ desc, ListPlan lp, const uint32_t* __restrict__ cand,
                const uint32_t* __restrict__ boff, int P, uint32_t max_w, int ignore_strand, int strand_filter,
                int32_t* __restrict__ cov, uint8_t* __restrict__ region_hit, LongIdx lg) {
    __shared__ __align__(16) int sm[WARPS][WT_ONE];
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;
    int* diff = sm[warp];
    const int64_t step = (int64_t)gridDim.x * WARPS;
    const int sh = 32 - P;
    const uint32_t pmask = (1u << P) - 1u;
    for (int64_t t = (int64_t)blockIdx.x * WARPS + warp; t < T; t += step) {
        const SpDesc d = sp_load_desc(desc + t);
        const int64_t a = lp.ptr[d.region], b = lp.ptr[d.region + 1];
        const int tlen = d.tlen, t0 = (int)d.cts, t1 = t0 + tlen;
        const bool rev = d.flags & 1u, simple = (d.flags & 2u) != 0;
        const int rows = (tlen + ROW - 1) / ROW;
        for (int k = 0; k < rows; k++) reinterpret_cast<int4*>(diff)[k * 32 + lane] = make_int4(0, 0, 0, 0);
        __syncwarp();
        int64_t qa = a, qb = b;              // last range with xoff <= t0
        while (qb - qa > 1) {
            const int64_t mid = (qa + qb) >> 1;
            if (__ldg(lp.xoff + mid) <= t0) qa = mid;
            else qb = mid;
        }
        bool hit = false;
        for (int64_t q = qa; q < b; q++) {
            const int xo = __ldg(lp.xoff + q);
            if (xo >= t1) break;
            const uint32_t s = __ldg(lp.xgs + q), e = __ldg(lp.xge + q);
            if (e + 1u == s) continue;
            const int w = (int)(e - s) + 1;
            const int k0 = max(xo, t0), k1 = min(xo + w, t1);              // stitched [k0, k1)
            if (k0 >= k1) continue;
            const uint32_t ps = s + (uint32_t)(k0 - xo), pe = s + (uint32_t)(k1 - 1 - xo);   // genomic piece
            const uint32_t first = ps >= max_w ? ps - max_w + 1u : 0u;
            const uint32_t c0 = __ldg(boff + (first >> SUB_SHIFT)), c1 = __ldg(boff + (pe >> SUB_SHIFT) + 1);
            // candidates 128 at a time: the four loads of a lane are in flight together, and the
            // next batch is requested before this one is used
            auto fetch = [&](uint32_t i0, uint32_t* wv) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t i = i0 + (uint32_t)k * 32u + lane;
                    wv[k] = i < c1 ? __ldg(cand + i) : 0u;          // 0: width 0, skipped below
                }
            };
            uint32_t wv[4], wn[4];
            if (c0 < c1) fetch(c0, wv);
            for (uint32_t i0 = c0; i0 < c1; i0 += 128) {
                if (i0 + 128 < c1) fetch(i0 + 128, wn);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t word = wv[k];
                    const int rel = ((int)((word - (ps & pmask)) << sh)) >> sh;
                    const uint32_t wd = word >> (STRANDED ? P + 2 : P);
                    if (wd == 0u) continue;
                    const int64_t rs64 = (int64_t)ps + rel;
                    const uint32_t rs = (uint32_t)rs64, re1 = rs + wd;
                    if (!(rs <= pe && re1 > ps)) continue;                     // does not reach the piece
                    int rst = 0;
                    if (STRANDED) {
                        const uint32_t cls = (word >> P) & 3u;
                        rst = cls == 0u ? 1 : (cls == 1u ? -1 : 0);
                    }
                    if (strand_filter != RCP_STRAND_ANY && rst != strand_filter) continue;
                    const int mult = sp_multiplicity(lp, a, b, q, simple, rs, re1, rst, ignore_strand, strand_filter);
                    if (mult == 0) continue;
                    hit = true;
                    // +mult on the covered part of the piece, in output order
                    const int ka = k0 + (int)(max(rs, ps) - ps) - t0;
                    const int kb1 = k0 + (int)(min(re1 - 1u, pe) - ps) + 1 - t0;    // may equal tlen
                    if (!rev) {
                        atomicAdd(diff + ka, mult);
                        if (kb1 < tlen) atomicSub(diff + kb1, mult);
                    } else {
                        atomicAdd(diff + (tlen - kb1), mult);
                        if (ka > 0) atomicSub(diff + (tlen - ka), mult);
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; k++) wv[k] = wn[k];
            }
        }
        if (lg.n) {             // the reads kept out of the binned index: whole reads against the element
            const uint2 lr = lp.lrange[d.region];
            for (uint32_t i = lr.x + lane; i < lr.y; i += 32) {
                const uint32_t rs = __ldg(lg.xs + i), re1 = __ldg(lg.e1 + i);
                const int rst = lg.st ? (int)__ldg(lg.st + i) : 0;
                if (strand_filter != RCP_STRAND_ANY && rst != strand_filter) continue;
                int mult = 0;
                for (int64_t z = a; z < b; z++) {
                    const uint32_t zs = __ldg(lp.xgs + z), ze = __ldg(lp.xge + z);
                    if (ze + 1u == zs) continue;
                    if (rs <= ze && re1 > zs &&
                        strand_ok(rst, lp.rstrand ? (int)__ldg(lp.rstrand + z) : 0, ignore_strand, strand_filter))
                        mult++;
                }
                if (mult == 0) continue;
                for (int64_t q = qa; q < b; q++) {
                    const int xo = __ldg(lp.xoff + q);
                    if (xo >= t1) break;
                    const uint32_t s = __ldg(lp.xgs + q), e = __ldg(lp.xge + q);
                    if (e + 1u == s || !(rs <= e && re1 > s)) continue;
                    const int pa = xo + (int)(max(rs, s) - s), pb = xo + (int)(min(re1 - 1u, e) - s);   // stitched, closed
                    if (pb < t0 || pa >= t1) continue;
                    const int ka = max(pa, t0) - t0, kb1 = min(pb, t1 - 1) + 1 - t0;
                    hit = true;
                    if (!rev) {
                        atomicAdd(diff + ka, mult);
                        if (kb1 < tlen) atomicSub(diff + kb1, mult);
                    } else {
                        atomicAdd(diff + (tlen - kb1), mult);
                        if (ka > 0) atomicSub(diff + (tlen - ka), mult);
                    }
                }
            }
        }
        hit = __any_sync(0xffffffffu, hit);
        __syncwarp();
        int32_t* dst = cov + d.out;
        switch (rows) {
            case 1: warp_scan_store_fwd<1>(diff, tlen, dst); break;
            case 2: warp_scan_store_fwd<2>(diff, tlen, dst); break;
            case 3: warp_scan_store_fwd<3>(diff, tlen, dst); break;
            case 4: warp_scan_store_fwd<4>(diff, tlen, dst); break;
            case 5: warp_scan_store_fwd<5>(diff, tlen, dst); break;
            case 6: warp_scan_store_fwd<6>(diff, tlen, dst); break;
            case 7: warp_scan_store_fwd<7>(diff, tlen, dst); break;
            default: {
                int pre = 0;
                for (int row = 0; row < rows; row++)
                    pre += warp_row_scan_store(diff + row * ROW, pre, 0, false, tlen - row * ROW, dst + row * ROW);
            }
        }
        if (hit && lane == 0) region_hit[d.region] = 1;
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
    }
}

// NULL rule (coverage.R:198,224-225): no overlapping read in any tile of the region.
__global__ void __launch_bounds__(CTA)
sp_null_kernel(int64_t R, const int32_t* __restrict__ plen, const uint8_t* __restrict__ region_hit,
               const uint32_t* __restrict__ cb, int32_t* __restrict__ len, uint8_t* __restrict__ is_null,
               unsigned long long* __restrict__ stats /* n_null, total_len, max_len, candidates */) {
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (r < R) {
        const bool null = plen[r] == 0 || region_hit[r] == 0;
        const int32_t out = null ? 0 : plen[r];
        len[r] = out;
        is_null[r] = null ? 1 : 0;
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
    if (r == 0) stats[3] = (unsigned long long)cb[NG] * CH;     // chunk capacity: >= the candidates
}

}  // namespace

// Same contract as coverage_ranges_bucketed.  RCP_SPLIT_NOT_APPLICABLE: the reads are too wide for
// the packed candidate word of this genome (or the genome too long for the shared-memory table);
// nothing has been produced and the caller uses another path.
struct DebugLap {
    bool on;
    std::chrono::steady_clock::time_point t0;
    explicit DebugLap() : on(getenv("RCP_DEBUG_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void lap(const char* what) {
        if (!on) return;
        cudaStreamSynchronize(g_ctx.stream);
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[rcp split] %-32s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t0).count());
        t0 = now;
    }
};

struct SortedCands {
    uint32_t* cand = nullptr;     // packed candidate words, sorted by 1-kb sub-bin
    uint32_t* boff = nullptr;     // n_groups * nb + 1 sub-bin offsets into cand
    uint32_t* cb = nullptr;       // NG + 1: chunk-list offsets per group (cb[NG] * CH >= candidates)
};

// split kernel + chunk lists + group sort.  tab: the mask's block table on the device.  The
// result lives in arena K (the caller keeps or drops it); B is scratch of the passes.
static int split_and_sort(ReadsIdx& rd, const uint32_t* tab, int words, int P, int n_groups, bool stranded,
                          bool st_arr, uint32_t max_pack_w, Arena& K, Arena& B, SortedCands* sc) {
    const int nb = 1 << (P - SUB_SHIFT);
    const uint32_t pmask = (1u << P) - 1u;
    const int split_grid = g_ctx.sm_count;
    const int sort_grid = 64;          // columns of the chunk-count table (one CTA each)
    const size_t pool_cap = (size_t)(rd.n / CH + 1) + (size_t)split_grid * NG +
                            (size_t)split_grid * (ST / 32) * SLAB * 2 + SLAB;
    RCP_TRY(K.reserve(Arena::pad(pool_cap * CH * 4) + Arena::pad((NG + 1) * 4) +
                      Arena::pad(((size_t)n_groups * nb + 1) * 4)));
    sc->cand = K.take<uint32_t>(pool_cap * CH);
    sc->cb = K.take<uint32_t>(NG + 1);
    sc->boff = K.take<uint32_t>((size_t)n_groups * nb + 1);
    RCP_TRY(B.reserve(Arena::pad(pool_cap * CH * 4) + Arena::pad(pool_cap * 2) + Arena::pad(pool_cap * 4) +
                      Arena::pad(16) + Arena::pad((size_t)sort_grid * NG * 4)));
    uint32_t* pool_next = B.take<uint32_t>(4);
    uint16_t* meta = B.take<uint16_t>(pool_cap);
    const size_t zero_b = B.used;
    uint32_t* pool = B.take<uint32_t>(pool_cap * CH);
    uint32_t* list = B.take<uint32_t>(pool_cap);
    uint32_t* col = B.take<uint32_t>((size_t)sort_grid * NG);
    if (B.used > B.cap || K.used > K.cap) return fail(RCP_ERR_CUDA, "internal: split arena overrun");
    DebugLap dbg;
    dbg.lap("  split_and_sort: arenas");
    {
        StageTimer t(ST_SP_SPLIT);
        RCP_CUDA(cudaMemsetAsync(B.base, 0, zero_b, g_ctx.stream));
        const size_t smem = sp_split_smem(words);
        SplitOut out = {pool, meta, pool_next};
        if (stranded) {     // no strand array: every read is '*'
            RCP_CUDA(cudaFuncSetAttribute(sp_split_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            sp_split_kernel<true><<<split_grid, ST, smem, g_ctx.stream>>>(rd.n, rd.g_start, rd.g_end1,
                                                                         st_arr ? rd.d_strand : nullptr, tab, words, P,
                                                                         max_pack_w, out);
        } else {
            RCP_CUDA(cudaFuncSetAttribute(sp_split_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            sp_split_kernel<false><<<split_grid, ST, smem, g_ctx.stream>>>(rd.n, rd.g_start, rd.g_end1, nullptr, tab,
                                                                          words, P, max_pack_w, out);
        }
        RCP_LAUNCHED();
    }
    dbg.lap("  split_and_sort: split kernel");
    {
        StageTimer t(ST_SP_SORT);
        {
            const uint16_t* a_meta = meta;
            const uint32_t* a_next = pool_next;
            void* args[] = {(void*)&a_meta, (void*)&a_next, (void*)&col, (void*)&sc->cb, (void*)&list};
            RCP_CUDA(cudaLaunchCooperativeKernel((const void*)sp_chunk_lists_kernel, dim3((unsigned)sort_grid), dim3(CS),
                                                 args, 0, g_ctx.stream));
            RCP_LAUNCHED();
        }
        dbg.lap("  split_and_sort: chunk lists");
        RCP_CUDA(cudaFuncSetAttribute(sp_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GSMEM));
        sp_group_kernel<<<n_groups, GT, GSMEM, g_ctx.stream>>>(pool, list, sc->cb, n_groups, nb, pmask, sc->cand,
                                                               sc->boff);
        RCP_LAUNCHED();
    }
    dbg.lap("  split_and_sort: group sort");
    return RCP_OK;
}

// The genome's split geometry: position bits of a candidate word, groups, table words.
struct SplitGeom {
    int words, P, n_groups, nb;
    uint32_t pmask;
    bool ok;
};
static SplitGeom split_geometry(const ReadsIdx& rd) {
    SplitGeom g;
    const int64_t span = (int64_t)rd.chrom_off[(size_t)rd.n_chrom];
    g.words = (int)((span >> (BLK_SHIFT + 4)) + 2);
    g.P = split_position_bits(span);
    g.n_groups = (int)std::max<int64_t>(1, (span + (1ll << g.P) - 1) >> g.P);
    g.nb = 1 << (g.P - SUB_SHIFT);
    g.pmask = (1u << g.P) - 1u;
    g.ok = g.n_groups <= NG && rd.n < 0x7ffffff0ll && sp_split_smem(g.words) <= SP_SMEM_MAX;
    return g;
}

// Builds the handle's binned index (every read, sorted by 1-kb bin).  RCP_SPLIT_NOT_APPLICABLE when
// the reads do not fit the packed word.  The words carry the strand class when the reads have one.
static LongIdx long_index(const ReadsIdx& rd) {
    LongIdx lg;
    lg.n = (uint32_t)rd.ln_n;
    lg.xs = rd.ln_xs;
    lg.e1 = rd.ln_e1;
    lg.st = rd.ln_st;
    lg.maxe1 = rd.ln_maxe1;
    return lg;
}

static int reads_build_binned(ReadsIdx& rd) {
    if (rd.bn_cand) return RCP_OK;
    DebugLap dbg;
    RCP_TRY(reads_resolve(rd));
    dbg.lap("binned: resolve reads");
    const SplitGeom g = split_geometry(rd);
    const bool stranded = rd.d_strand != nullptr;
    const int wbits = 32 - g.P - (stranded ? 2 : 0);
    if (!g.ok || wbits < 7) return RCP_SPLIT_NOT_APPLICABLE;
    // the words hold reads up to max_pack_w wide; wider ones go to the long-read list
    const uint32_t max_pack_w = std::min<uint32_t>((1u << wbits) - 1u, 8191u);
    rd.bn_max_pack_w = max_pack_w;
    if (rd.max_width > max_pack_w) {
        // how many: counted by the map kernel when the threshold it was given is this one
        // (a stranded handle, or a strandless one: the same rule on both sides)
        if (rd.long_thr != max_pack_w) return RCP_SPLIT_NOT_APPLICABLE;
        // a sample made of long reads is not what this index is for
        if (rd.n_long > rd.n / 8) return RCP_SPLIT_NOT_APPLICABLE;
        const size_t n = (size_t)rd.n_long;
        uint32_t* idx = nullptr;
        unsigned int* d_cur = nullptr;
        RCP_TRY(dalloc(&d_cur, 1));
        RCP_CUDA(cudaMemsetAsync(d_cur, 0, 4, g_ctx.stream));
        RCP_TRY(dalloc(&rd.ln_xs, n));
        RCP_TRY(dalloc(&rd.ln_e1, n));
        RCP_TRY(dalloc(&rd.ln_maxe1, n));
        if (rd.d_strand) RCP_TRY(dalloc(&rd.ln_st, n));
        RCP_TRY(dalloc(&idx, n));
        sp_long_collect_kernel<<<(unsigned)blocks_for(rd.n, LONG_PER), CTA, 0, g_ctx.stream>>>(
            rd.n, rd.g_start, rd.g_end1, max_pack_w, d_cur, (uint32_t)n, rd.ln_xs, idx);
        RCP_LAUNCHED();
        dfree(d_cur);
        dbg.lap("  long: collect");
        RCP_TRY(sort_pairs_u32(rd.ln_xs, idx, (int64_t)n, rd.key_bits));
        dbg.lap("  long: sort");
        if (n > 0) {
            sp_long_gather_kernel<<<blocks_for((int64_t)n, CTA), CTA, 0, g_ctx.stream>>>((uint32_t)n, idx, rd.g_end1,
                                                                                        rd.d_strand, rd.ln_e1, rd.ln_st);
            RCP_LAUNCHED();
        }
        RCP_TRY(running_max_u32_device(rd.ln_e1, rd.ln_maxe1, (int64_t)n));
        rd.ln_n = (int64_t)n;
        dfree(idx);
        dbg.lap("binned: long-read list");
    }
    Arena K, B, Tb;
    RCP_TRY(Tb.reserve(Arena::pad((size_t)g.words * 4)));
    uint32_t* tab = Tb.take<uint32_t>((size_t)g.words);
    RCP_CUDA(cudaMemsetAsync(tab, 0xff, (size_t)g.words * 4, g_ctx.stream));      // the mask "everything"
    SortedCands sc;
    RCP_TRY(split_and_sort(rd, tab, g.words, g.P, g.n_groups, stranded, stranded, max_pack_w, K, B, &sc));
    rd.bn_base = K.base;
    K.base = nullptr;                   // the handle owns it now
    rd.bn_cand = sc.cand;
    rd.bn_boff = sc.boff;
    rd.bn_cb = sc.cb;
    rd.bn_P = g.P;
    rd.bn_stranded = stranded;
    dbg.lap("binned: split + sort");
    return RCP_OK;
}

// fz != nullptr: the FUSED form (rcp_coverage_profile): no coverage is stored, the tiles add their
// bin sums to accumulators and sp_bins_finish_kernel writes the matrix (cv is scratch then).
// RCP_SPLIT_NOT_APPLICABLE there also when the windows differ in length or are shorter than the
// bin count (interpolation): the caller composes the two stages instead.
struct FusedReq {
    int n_bins, seed, sample_kind;
    double scale;
    double* d_out;
    int64_t ld;
    uint8_t* d_is_null;      // may be nullptr
};

static int split_impl(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                      const int32_t* end, const int8_t* strand, int ignore_strand,
                      int strand_filter, int mem, Coverage* cv, const FusedReq* fz) {
    const bool stranded = !((strand_filter == RCP_STRAND_ANY) && (ignore_strand || strand == nullptr));
    const bool st_arr = stranded && rd.d_strand != nullptr;      // strandless reads are all '*'
    if (rd.failed != RCP_OK) return reads_finish(rd);              // a deferred load that failed
    const int64_t span = (int64_t)rd.chrom_off[(size_t)rd.n_chrom];
    const int words = (int)((span >> (BLK_SHIFT + 4)) + 2);
    const int P = split_position_bits(span);
    const int n_groups = (int)std::max<int64_t>(1, (span + (1ll << P) - 1) >> P);
    const int wbits = 32 - P - (stranded ? 2 : 0);
    if (n_groups > NG || rd.n >= 0x7ffffff0ll || sp_split_smem(words) > SP_SMEM_MAX)
        return RCP_SPLIT_NOT_APPLICABLE;
    const bool have_index = rd.bn_cand && rd.bn_P == P && (rd.bn_stranded || !stranded);
    if (!have_index && !rd.pending && (rd.max_width > 8191u || rd.max_width >= (1u << wbits)))
        return RCP_SPLIT_NOT_APPLICABLE;
    const uint32_t pmask = (1u << P) - 1u;

    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_chrom.init(chrom, (size_t)R, mem));
    RCP_TRY(d_start.init(start, (size_t)R, mem));
    RCP_TRY(d_end.init(end, (size_t)R, mem));
    RCP_TRY(d_strand.init(strand, (size_t)R, mem));

    // ---- plan -------------------------------------------------------------------------------
    Arena A;
    const size_t r = (size_t)R;
    RCP_TRY(A.reserve(Arena::pad(64) + Arena::pad((size_t)words * 4) + Arena::pad(r * 4) * 2 + Arena::pad(r) * 2 +
                      Arena::pad(r * 8) * 2 + Arena::pad((r + 1) * 8)));
    // zero-initialised block first (ONE memset): status words, block table, region hit flags
    unsigned int* err = A.take<unsigned int>(16);         // [0] err; pstats at +16 bytes
    unsigned long long* pstats = reinterpret_cast<unsigned long long*>(err + 4);   // [0] total len [1] max len [2] 2^32 - min len
    uint32_t* tab = A.take<uint32_t>((size_t)words);
    uint8_t* region_hit = A.take<uint8_t>(r);
    const size_t zero_bytes = A.used;
    uint32_t* gs = A.take<uint32_t>(r);
    int32_t* plen = A.take<int32_t>(r);
    uint8_t* flags = A.take<uint8_t>(r);
    int64_t* ntile = A.take<int64_t>(r);
    int64_t* padded = A.take<int64_t>(r);
    int64_t* off_tile = A.take<int64_t>(r + 1);
    if (A.used > A.cap) return fail(RCP_ERR_CUDA, "internal: split plan arena overrun");

    cv->n_regions = R;
    RCP_TRY(dalloc(&cv->off, r + 1));
    RCP_TRY(dalloc(&cv->len, r));
    RCP_TRY(dalloc(&cv->is_null, r));
    RCP_TRY(dalloc(&cv->d_stats, 5));
    auto give_up = [&]() {
        dfree(cv->off);
        dfree(cv->len);
        dfree(cv->is_null);
        dfree(cv->d_stats);
        return RCP_SPLIT_NOT_APPLICABLE;
    };
    {
        StageTimer t(ST_SP_PLAN);
        RCP_CUDA(cudaMemsetAsync(A.base, 0, zero_bytes, g_ctx.stream));
        if (R == 0) RCP_CUDA(cudaMemsetAsync(cv->d_stats, 0, 40, g_ctx.stream));     // else: sp_plan_kernel
        if (R > 0) {
            sp_plan_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(
                R, d_chrom.ptr, d_start.ptr, d_end.ptr, d_strand.ptr, rd.d_chrom_off, rd.d_chrom_len,
                rd.n_chrom, ignore_strand, strand_filter, gs, plen, flags, ntile, padded, tab, err,
                pstats, cv->d_stats);
            RCP_LAUNCHED();
        }
        RCP_TRY(exclusive_scan2_i64(ntile, off_tile, off_tile + R, padded, cv->off, cv->off + R, R));
    }
    struct Host {
        int64_t T, total_padded;
        unsigned long long pstats[3];
        unsigned int err;
    } h = {0, 0, {0, 0, 0}, 0};
    // The read passes do not depend on anything the host is about to learn: they are queued
    // BEFORE the host waits for the plan's numbers, so the GPU works through the round trip.  (A
    // sample whose reads turn out not to fit the packed word is caught below; the passes have
    // written into their own arenas only.)
    Arena K, B;
    SortedCands sc;
    {
        FetchItem items[8] = {{off_tile + R, &h.T, 8}, {cv->off + R, &h.total_padded, 8}, {pstats, h.pstats, 24},
                              {err, &h.err, 4}};
        int n_items = 4;
        reads_pending_items(rd, items, &n_items);       // a deferred rcp_reads_load is validated here
        RCP_TRY(fetch_begin(items, n_items));
        if (!have_index) RCP_TRY(split_and_sort(rd, tab, words, P, n_groups, stranded, st_arr, 0xffffffffu, K, B, &sc));
        RCP_TRY(fetch_end(items, n_items));
        RCP_TRY(reads_finish(rd));
    }
    if (h.err & 1u) return fail(RCP_ERR_DATA, "a region has a chromosome id outside [0, n_chrom)");
    if (h.err & 2u) return fail(RCP_ERR_DATA, "a region has end < start - 1");
    const int64_t T = h.T;
    if (T > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 coverage tiles");
    // (with the handle's binned index the words hold the reads up to bn_max_pack_w; wider ones
    // come from the long-read list)
    const uint32_t max_w = have_index ? std::max(1u, std::min(rd.max_width, rd.bn_max_pack_w))
                                      : (rd.max_width > 0 ? rd.max_width : 1u);
    if (!have_index && (max_w > 8191u || max_w >= (1u << wbits))) return give_up();

    // ---- fused: one common window length, bin edges of splitVector (util.R:74-80) -------------
    FusedBins fb = {nullptr, 0, R, nullptr};
    Arena F;
    if (fz) {
        const int64_t max_len = (int64_t)h.pstats[1];
        const int64_t min_len = h.pstats[2] ? 0x100000000ll - (int64_t)h.pstats[2] : 0;
        const int n = fz->n_bins;
        if (max_len != min_len || (max_len > 0 && max_len < n)) return give_up();
        const int64_t Lc = max_len > 0 ? max_len : n;       // no valid window at all: any layout
        std::vector<int32_t> edge((size_t)n + 1);
        {
            std::vector<int> perm((size_t)n), scratch((size_t)n), rank((size_t)n);
            RRng* rng = new RRng;
            rng->seed((uint32_t)fz->seed, fz->sample_kind);
            rng->sample(n, n, scratch.data(), perm.data());
            delete rng;
            for (int pos = 0; pos < n; pos++) rank[(size_t)perm[(size_t)pos] - 1] = pos + 1;
            const int64_t b = Lc / n, d = Lc - b * n;
            int64_t at = 0;
            for (int i = 0; i < n; i++) {
                edge[(size_t)i] = (int32_t)at;
                at += b + (rank[(size_t)i] <= d ? 1 : 0);
            }
            edge[(size_t)n] = (int32_t)at;
        }
        RCP_TRY(F.reserve(Arena::pad(((size_t)n + 1) * 4) + Arena::pad((size_t)n * r * 8)));
        int32_t* d_edge = F.take<int32_t>((size_t)n + 1);
        fb.acc = F.take<unsigned long long>((size_t)n * r);
        RCP_CUDA(cudaMemcpyAsync(d_edge, edge.data(), ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, g_ctx.stream));
        RCP_CUDA(cudaMemsetAsync(fb.acc, 0, (size_t)n * r * 8, g_ctx.stream));
        fb.edge = d_edge;
        fb.n = n;
    } else {
        cv->path = RCP_PATH_SPLIT;
        cv->total_padded = h.total_padded;
        cv->total_len = (int64_t)h.pstats[0];       // upper bounds until the NULL rule has run
        cv->max_len = (int32_t)h.pstats[1];
        cv->n_null = 0;
        cv->stats_pending = true;
        // 4 bytes per element: the storage width is decided on the device, after this allocation
        RCP_TRY(dalloc(&cv->cov, (size_t)h.total_padded));
        if (getenv("RCP_COVERAGE_WIDE") == nullptr) cv->d_bound = cv->d_stats + 4;
    }
    unsigned long long* bound = cv->d_bound ? cv->d_stats + 4 : nullptr;     // nullptr: int32 storage

    // ---- the sorted candidates: the handle's binned index when it has one, else this mask's ----
    bool words_stranded = stranded;
    if (have_index) {
        sc.cand = rd.bn_cand;
        sc.boff = rd.bn_boff;
        sc.cb = rd.bn_cb;
        words_stranded = rd.bn_stranded;
    }
    uint32_t* cand = sc.cand;
    uint32_t* boff = sc.boff;
    uint32_t* cb = sc.cb;
    LongIdx lg = long_index(rd);
    if (!have_index) lg.n = 0;
    Arena D;
    RCP_TRY(D.reserve(Arena::pad((size_t)(T + 1) * sizeof(SpDesc)) + (lg.n ? Arena::pad((size_t)(T + 1) * 4) +
                                                                            Arena::pad((size_t)(T + 1) * 8) : 0)));
    SpDesc* desc = D.take<SpDesc>((size_t)T + 1);
    uint32_t* tabs = lg.n ? D.take<uint32_t>((size_t)T + 1) : nullptr;
    uint2* lrange = lg.n ? D.take<uint2>((size_t)T + 1) : nullptr;
    if (T > 0) {
        StageTimer t(ST_SP_PLAN);
        sp_tiles_kernel<<<blocks_for(T, CTA), CTA, 0, g_ctx.stream>>>(R, T, off_tile, gs, plen, flags,
                                                                     fz ? nullptr : cv->off, fb.edge, fb.n, max_w, pmask, boff,
                                                                     desc, tabs,
                                                                     lg.xs, lg.maxe1, lg.n, lrange, bound);
        RCP_LAUNCHED();
    }
    if (T > 0) {
        {
            StageTimer t(fz ? ST_FUSED : ST_SP_TILE);
            const int64_t want = blocks_for(T, WARPS);
            auto launch = [&](auto kern) -> int {
                int per_sm = 0;
                RCP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WTILE_SMEM));
                RCP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, CTA, WTILE_SMEM));
                per_sm = std::max(per_sm, 1);
                kern<<<(unsigned)std::min<int64_t>(want, (int64_t)g_ctx.sm_count * per_sm), CTA, WTILE_SMEM,
                       g_ctx.stream>>>(
                    T, desc, cand, P, cv->cov, region_hit, fb, lg, tabs, lrange, bound);
                RCP_LAUNCHED();
                return RCP_OK;
            };
            if (fz) RCP_TRY(words_stranded ? launch(sp_wtile_kernel<true, true>) : launch(sp_wtile_kernel<false, true>));
            else RCP_TRY(words_stranded ? launch(sp_wtile_kernel<true, false>) : launch(sp_wtile_kernel<false, false>));
        }
    }
    if (fz) {
        if (R > 0) {
            StageTimer t(ST_FUSED);
            sp_bins_finish_kernel<<<dim3(blocks_for(R, CTA), (unsigned)fb.n), CTA, 0, g_ctx.stream>>>(
                fb, plen, region_hit, fz->scale, fz->d_out, fz->ld, fz->d_is_null);
            RCP_LAUNCHED();
        }
        return RCP_OK;
    }
    if (R > 0) {
        StageTimer t(ST_SP_PLAN);
        sp_null_kernel<<<blocks_for(R, CTA), CTA, 0, g_ctx.stream>>>(R, plen, region_hit, cb, cv->len, cv->is_null,
                                                                    cv->d_stats);
        RCP_LAUNCHED();
    }
    return RCP_OK;
}

int coverage_ranges_split(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                          const int32_t* end, const int8_t* strand, int ignore_strand,
                          int strand_filter, int mem, Coverage* cv) {
    return split_impl(rd, R, chrom, start, end, strand, ignore_strand, strand_filter, mem, cv, nullptr);
}

// coverageRef + profileMatrix of equal-length windows WITHOUT storing the coverage (d_out, d_is_null:
// device memory).  RCP_SPLIT_NOT_APPLICABLE: compose rcp_coverage + rcp_profile_matrix instead.
int coverage_profile_split(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                           const int32_t* end, const int8_t* strand, int ignore_strand,
                           int strand_filter, int mem, int n_bins, int seed, int sample_kind,
                           double scale, double* d_out, int64_t ld, uint8_t* d_is_null) {
    if (n_bins < 1 || n_bins > 30000) return RCP_SPLIT_NOT_APPLICABLE;
    Coverage scratch;
    const FusedReq fz = {n_bins, seed, sample_kind, scale, d_out, ld, d_is_null};
    const int rc = split_impl(rd, R, chrom, start, end, strand, ignore_strand, strand_filter, mem, &scratch, &fz);
    coverage_release(scratch);
    return rc;
}

// rcp_coverage_list through the handle's binned index (built here on first use: coverageRnaRef
// makes three coverage calls per sample on the same reads).  RCP_SPLIT_NOT_APPLICABLE: the reads do
// not fit the packed word; the caller uses the sorted-pair path.
int coverage_list_split(ReadsIdx& rd, int64_t G, const int64_t* ptr, int64_t n_ranges, const int32_t* chrom,
                        const int32_t* start, const int32_t* end, const int8_t* strand, int ignore_strand,
                        int strand_filter, int mem, Coverage* cv) {
    DebugLap dbg;
    {
        const int rc = reads_build_binned(rd);
        if (rc != RCP_OK) return rc;
    }
    dbg.lap("list: binned index");
    const SplitGeom g = split_geometry(rd);
    const uint32_t max_w = std::max(1u, std::min(rd.max_width, rd.bn_max_pack_w));
    const LongIdx lg = long_index(rd);
    DevIn<int64_t> d_ptr;
    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_ptr.init(ptr, (size_t)G + 1, mem));
    RCP_TRY(d_chrom.init(chrom, (size_t)n_ranges, mem));
    RCP_TRY(d_start.init(start, (size_t)n_ranges, mem));
    RCP_TRY(d_end.init(end, (size_t)n_ranges, mem));
    RCP_TRY(d_strand.init(strand, (size_t)n_ranges, mem));
    Arena A;
    const size_t r = (size_t)G, nr = (size_t)n_ranges;
    RCP_TRY(A.reserve(Arena::pad(64) + Arena::pad(r) * 2 + Arena::pad(r * 4) + Arena::pad(r * 8) * 3 +
                      Arena::pad((r + 1) * 8) + Arena::pad(nr * 4) * 3));
    unsigned int* err = A.take<unsigned int>(16);
    unsigned long long* pstats = reinterpret_cast<unsigned long long*>(err + 4);
    uint8_t* region_hit = A.take<uint8_t>(r);
    const size_t zero_bytes = A.used;
    uint8_t* flags = A.take<uint8_t>(r);
    int32_t* plen = A.take<int32_t>(r);
    int64_t* ntile = A.take<int64_t>(r);
    int64_t* padded = A.take<int64_t>(r);
    int64_t* off_tile = A.take<int64_t>(r + 1);
    ListPlan lp;
    lp.ptr = d_ptr.ptr;
    lp.rstrand = d_strand.ptr;
    lp.xgs = A.take<uint32_t>(nr);
    lp.xge = A.take<uint32_t>(nr);
    lp.xoff = A.take<int32_t>(nr);
    lp.lrange = A.take<uint2>(r);
    if (A.used > A.cap) return fail(RCP_ERR_CUDA, "internal: list plan arena overrun");
    cv->n_regions = G;
    RCP_TRY(dalloc(&cv->off, r + 1));
    RCP_TRY(dalloc(&cv->len, r));
    RCP_TRY(dalloc(&cv->is_null, r));
    RCP_TRY(dalloc(&cv->d_stats, 4));
    struct Host {
        int64_t T, total_padded;
        unsigned long long pstats[2];
        unsigned int err;
    } h = {0, 0, {0, 0}, 0};
    {
        StageTimer t(ST_COV_LIST);
        RCP_CUDA(cudaMemsetAsync(A.base, 0, zero_bytes, g_ctx.stream));
        RCP_CUDA(cudaMemsetAsync(cv->d_stats, 0, 32, g_ctx.stream));
        if (G > 0) {
            sp_list_plan_kernel<<<blocks_for(G, CTA), CTA, 0, g_ctx.stream>>>(
                G, lp, d_chrom.ptr, d_start.ptr, d_end.ptr, rd.d_chrom_off, rd.d_chrom_len, rd.n_chrom, plen, flags,
                ntile, padded, err, pstats, lg);
            RCP_LAUNCHED();
        }
        RCP_TRY(exclusive_scan2_i64(ntile, off_tile, off_tile + G, padded, cv->off, cv->off + G, G));
        const FetchItem items[4] = {{off_tile + G, &h.T, 8}, {cv->off + G, &h.total_padded, 8}, {pstats, h.pstats, 16},
                                    {err, &h.err, 4}};
        RCP_TRY(fetch_and_sync(items, 4));
    }
    dbg.lap("list: plan + fetch");
    if (h.err & 1u) return fail(RCP_ERR_DATA, "a range has a chromosome id outside [0, n_chrom)");
    if (h.err & 2u) return fail(RCP_ERR_DATA, "a range has end < start - 1");
    if (h.err & 4u) return fail(RCP_ERR_DATA, "the ranges of one list element lie on different chromosomes");
    const int64_t T = h.T;
    if (T > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 coverage tiles");
    cv->path = 0;
    cv->total_padded = h.total_padded;
    cv->total_len = (int64_t)h.pstats[0];
    cv->max_len = (int32_t)h.pstats[1];
    cv->n_null = 0;
    cv->stats_pending = true;
    RCP_TRY(dalloc(&cv->cov, (size_t)h.total_padded));
    Arena D;
    RCP_TRY(D.reserve(Arena::pad((size_t)(T + 1) * sizeof(SpDesc))));
    SpDesc* desc = D.take<SpDesc>((size_t)T + 1);
    StageTimer t(ST_COV_LIST);
    if (T > 0) {
        sp_list_tiles_kernel<<<blocks_for(T, CTA), CTA, 0, g_ctx.stream>>>(G, T, off_tile, plen, flags, cv->off, desc);
        RCP_LAUNCHED();
        const unsigned grid = (unsigned)std::min<int64_t>(blocks_for(T, WARPS), (int64_t)g_ctx.sm_count * 4);
        if (rd.bn_stranded)
            sp_ltile_kernel<true><<<grid, CTA, 0, g_ctx.stream>>>(T, desc, lp, rd.bn_cand, rd.bn_boff, g.P, max_w,
                                                                 ignore_strand, strand_filter, cv->cov, region_hit, lg);
        else
            sp_ltile_kernel<false><<<grid, CTA, 0, g_ctx.stream>>>(T, desc, lp, rd.bn_cand, rd.bn_boff, g.P, max_w,
                                                                  ignore_strand, strand_filter, cv->cov, region_hit, lg);
        RCP_LAUNCHED();
    }
    if (G > 0) {
        sp_null_kernel<<<blocks_for(G, CTA), CTA, 0, g_ctx.stream>>>(G, plen, region_hit, rd.bn_cb, cv->len, cv->is_null,
                                                                    cv->d_stats);
        RCP_LAUNCHED();
    }
    dbg.lap("list: tiles");
    return RCP_OK;
}

}  // namespace rcp
