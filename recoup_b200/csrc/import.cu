// Read import, the decode half (SURVEY 8f N3): what readBam / readBed of the reference
// (/root/reference/R/ranges.R:111-146) hand to the hot path, produced on the device.
//
//   BAM   readGAlignments(file) then as(., "GRanges") (spliceAction keep / remove) or
//         unlist(grglist(.)) (spliceAction split), then trim().  The caller inflates the BGZF
//         blocks (host zlib) and passes the alignment-record section; the record chain is walked
//         once on the host (rcp_bam_index: the records are length-prefixed), everything else -- flag
//         filter, CIGAR walk, N-split, trim, compaction -- is one thread per record on the device.
//   BED   trim(import.bed(file, trackLine = FALSE)): text lines -> chrom id, start + 1, end, strand.
//         Line starts by a counting pass + prefix sum over the bytes, then one thread per line.
//
// Both run count -> prefix sum -> write, so that the output keeps the file order (the seeded
// down-sampling of preprocessRanges indexes the reads by position).  The result stays on the
// device behind a `decoded` handle: rcp_reads_load_decoded feeds it to the hot path without a
// host round trip, rcp_decoded_fetch hands the arrays back.
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include <algorithm>

#include "cov_common.cuh"
#include "rcp_internal.cuh"

namespace rcp {

using namespace covk;

namespace {

struct Decoded {
    int64_t n = 0;
    int32_t* chrom = nullptr;
    int32_t* start = nullptr;
    int32_t* end = nullptr;
    int8_t* strand = nullptr;
};
std::map<int, std::unique_ptr<Decoded>> g_decoded;
int g_next_decoded = 1 << 20;

void decoded_release(Decoded& d) {
    dfree(d.chrom);
    dfree(d.start);
    dfree(d.end);
    dfree(d.strand);
    d.n = 0;
}

struct Out {
    int32_t* chrom;
    int32_t* start;
    int32_t* end;
    int8_t* strand;
};

__device__ __forceinline__ uint32_t ld_u32(const uint8_t* __restrict__ p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ uint32_t ld_u16(const uint8_t* __restrict__ p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8);
}

// trim() of a GRanges with known seqlengths: [max(start, 1), min(end, L)]; a range that lies
// wholly outside becomes the zero-width range at the boundary it left by
__device__ __forceinline__ void trim_range(int64_t s, int64_t e, int64_t L, int32_t* so, int32_t* eo) {
    int64_t s2 = max(s, (int64_t)1), e2 = min(e, L);
    if (e2 < s2 - 1) {
        if (s > L) {
            s2 = L + 1;
            e2 = L;
        } else {
            e2 = s2 - 1;
        }
    }
    *so = (int32_t)s2;
    *eo = (int32_t)e2;
}

// ------------------------------------------------------------------------------- BAM ----------
// err bits: 1 record chain / truncated record, 2 refID outside the header's references,
//           4 CIGAR operation code > 8, 8 mapped record without a CIGAR,
//           16 (tagFilter) an aux field runs past its record or has an unknown type,
//           32 (which) the records are not sorted by (refID, POS)

// The ScanBamParam filters of rcp_bam_decode_param.  The tag table -- n_tags Tag entries, the
// int64 values of the integer tags, n_str + 1 offsets of the string values, their bytes -- is
// staged in shared memory by every CTA of the kernels that read it.
struct Tag {
    uint32_t name;      // the two characters, the first in the low byte
    uint32_t is_str;    // 0: the values are integers, 1: strings
    uint32_t v0, v1;    // the accepted values: [v0, v1) of the integers or of the strings
};
struct Filter {
    uint32_t keep0, keep1;  // bamFlag(param, asInteger = TRUE)
    int mapq_min;           // < 0: no MAPQ filter
    int simple_cigar;
    int n_tags;             // <= 32
    int n_int, n_str;
    int table_words;        // size of the tag table in uint32 words
    const uint32_t* table;  // device
};

__device__ __forceinline__ int64_t aux_int(const uint8_t* p, uint8_t ty) {
    switch (ty) {
        case 'c': return (int8_t)p[0];
        case 'C': return p[0];
        case 's': return (int16_t)ld_u16(p);
        case 'S': return ld_u16(p);
        case 'i': return (int32_t)ld_u32(p);
        default: return ld_u32(p);      // 'I'
    }
}

// tagFilter over the aux fields [q, end) of the record at p (SAMv1 4.2.4): 1 every filter tag is
// present with one of its accepted values, 0 not, -1 a field runs past the record or has an
// unknown type.  Every field is walked, so malformed aux data is reported whatever the filter.
// Integer values match c C s S i I fields, string values Z and A fields; the first occurrence of
// a tag decides.
__device__ __forceinline__ int tags_pass(const uint8_t* __restrict__ p, int64_t q, int64_t end, const Filter& f,
                         const uint32_t* tab) {
    const Tag* tags = reinterpret_cast<const Tag*>(tab);
    const long long* ival = reinterpret_cast<const long long*>(tab + 4 * f.n_tags);
    const uint32_t* soff = tab + 4 * f.n_tags + 2 * f.n_int;
    const uint8_t* sbytes = reinterpret_cast<const uint8_t*>(soff + f.n_str + 1);
    uint32_t seen = 0, ok = 0;
    while (q < end) {
        if (end - q < 3) return -1;
        const uint32_t name = ld_u16(p + q);
        const uint8_t ty = p[q + 2];
        q += 3;
        int64_t sz;
        int kind = 0;       // 1 integer, 2 string, 0 neither
        switch (ty) {
            case 'A': sz = 1; kind = 2; break;
            case 'c': case 'C': sz = 1; kind = 1; break;
            case 's': case 'S': sz = 2; kind = 1; break;
            case 'i': case 'I': sz = 4; kind = 1; break;
            case 'f': sz = 4; break;
            case 'Z': case 'H': {
                int64_t z = q;
                while (z < end && p[z] != 0) z++;
                if (z >= end) return -1;
                sz = z + 1 - q;
                kind = ty == 'Z' ? 2 : 0;
                break;
            }
            case 'B': {
                if (end - q < 5) return -1;
                const uint8_t sub = p[q];
                const int es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2
                             : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
                if (es == 0) return -1;
                sz = 5 + (int64_t)ld_u32(p + q + 1) * es;
                break;
            }
            default: return -1;
        }
        if (sz > end - q) return -1;
        for (int k = 0; k < f.n_tags; k++) {
            if (tags[k].name != name || ((seen >> k) & 1u)) continue;
            seen |= 1u << k;
            bool hit = false;
            if (kind == 1 && !tags[k].is_str) {
                const int64_t v = aux_int(p + q, ty);
                for (uint32_t j = tags[k].v0; j < tags[k].v1 && !hit; j++) hit = ival[j] == v;
            } else if (kind == 2 && tags[k].is_str) {
                const uint32_t len = ty == 'A' ? 1u : (uint32_t)(sz - 1);
                for (uint32_t j = tags[k].v0; j < tags[k].v1 && !hit; j++) {
                    if (soff[j + 1] - soff[j] != len) continue;
                    hit = true;
                    for (uint32_t b = 0; b < len && hit; b++) hit = sbytes[soff[j] + b] == p[q + b];
                }
            }
            if (hit) ok |= 1u << k;
        }
        q += sz;
    }
    return ok == (f.n_tags == 32 ? ~0u : (1u << f.n_tags) - 1u);
}

// One alignment record [o, o1) of rec: returns the ranges it yields (0 when it is unmapped,
// malformed or, FILTER, dropped by the filters), writes them from out[w] on when WRITE, and its
// reference span (M D N = X; 0 for a CIGAR that takes no reference) into span.  Every mapped
// record is checked for errors, whether the filters keep it or not.
template <bool WRITE, bool FILTER>
__device__ __forceinline__ uint32_t bam_record(const uint8_t* __restrict__ rec, int64_t n_bytes, int64_t o, int64_t o1,
                                               int n_ref, const int64_t* __restrict__ ref_len, int split, uint32_t w,
                                               Out out, unsigned int* __restrict__ err, const Filter& f,
                                               const uint32_t* tab, int64_t& span) {
    uint32_t cnt = 0;
    do {
        if (o < 0 || o1 > n_bytes || o1 - o < 36) {
            atomicOr(err, 1u);
            break;
        }
        const uint8_t* p = rec + o;
        if ((int64_t)ld_u32(p) + 4 != o1 - o) {
            atomicOr(err, 1u);
            break;
        }
        const int ref = (int)ld_u32(p + 4), pos = (int)ld_u32(p + 8);
        const uint32_t l_name = p[12], n_cig = ld_u16(p + 16), flag = ld_u16(p + 18);
        if ((flag & 4u) || ref < 0 || pos < 0) break;          // unmapped: readGAlignments drops it
        if (ref >= n_ref) {
            atomicOr(err, 2u);
            break;
        }
        if (n_cig == 0) {
            atomicOr(err, 8u);
            break;
        }
        const int64_t cig = 36 + (int64_t)l_name;
        if (cig + 4 * (int64_t)n_cig > o1 - o) {
            atomicOr(err, 1u);
            break;
        }
        bool pass = true;
        if (FILTER) {
            pass = (((flag & f.keep1) | (~flag & f.keep0)) & 0xfffu) == 0xfffu &&
                   (f.mapq_min < 0 || (int)p[13] >= f.mapq_min);
            if (f.simple_cigar) pass = pass && n_cig == 1 && (ld_u32(p + cig) & 15u) == 0u;
            if (f.n_tags > 0) {
                const int64_t l_seq = (int32_t)ld_u32(p + 20);
                const int64_t aux = cig + 4 * (int64_t)n_cig + (l_seq + 1) / 2 + l_seq;
                const int t = (l_seq < 0 || aux > o1 - o) ? -1 : tags_pass(p, aux, o1 - o, f, tab);
                if (t < 0) {
                    atomicOr(err, 16u);
                    break;
                }
                pass = pass && t == 1;
            }
            if (WRITE && !pass) break;
        }
        const int64_t L = ref_len[ref];
        const int8_t st = (flag & 16u) ? -1 : 1;
        int64_t cur = (int64_t)pos + 1, blk = 0;          // open block [cur, cur + blk)
        bool bad = false;
        auto emit = [&]() {
            if (WRITE) {
                trim_range(cur, cur + blk - 1, L, out.start + w, out.end + w);
                out.chrom[w] = ref;
                out.strand[w] = st;
                w++;
            }
            cnt++;
        };
        for (uint32_t k = 0; k < n_cig; k++) {
            const uint32_t c = ld_u32(p + cig + 4 * k), op = c & 15u;
            const int64_t len = (int64_t)(c >> 4);
            if (op > 8u) bad = true;
            if (op == 0u || op == 2u || op == 7u || op == 8u) {      // M D = X
                blk += len;
            } else if (op == 3u) {                                      // N
                if (split) {
                    if (blk > 0) emit();
                    cur += blk + len;
                    blk = 0;
                } else {
                    blk += len;
                }
            }
        }
        if (bad) {
            atomicOr(err, 4u);
            cnt = 0;
            break;
        }
        // as(., "GRanges") keeps an alignment of reference width 0; grglist drops empty ranges
        if (blk > 0 || !split) emit();
        span = cur + blk - ((int64_t)pos + 1);
        if (FILTER && !pass) cnt = 0;
    } while (false);
    return cnt;
}

template <bool FILTER>
__device__ __forceinline__ void stage_tag_table(const Filter& f, uint32_t* s_tab) {
    if (FILTER && f.table_words > 0) {
        for (int i = threadIdx.x; i < f.table_words; i += CTA) s_tab[i] = f.table[i];
        __syncthreads();
    }
}

// One thread per alignment record, output in file order.  WRITE = false: counts[r] = ranges the
// record yields; WRITE = true: they go to out[where[r]...].
template <bool WRITE, bool FILTER>
__global__ void __launch_bounds__(CTA)
bam_records_kernel(const uint8_t* __restrict__ rec, int64_t n_bytes, const int64_t* __restrict__ off, int64_t n,
                   int n_ref, const int64_t* __restrict__ ref_len, int split, uint32_t* __restrict__ counts,
                   const uint32_t* __restrict__ where, Out out, unsigned int* __restrict__ err, Filter f) {
    extern __shared__ __align__(16) uint32_t s_tab[];
    stage_tag_table<FILTER>(f, s_tab);
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (r >= n) return;
    int64_t span;
    const uint32_t cnt = bam_record<WRITE, FILTER>(rec, n_bytes, off[r], off[r + 1], n_ref, ref_len, split,
                                                   WRITE ? where[r] : 0u, out, err, f, s_tab, span);
    if (!WRITE) counts[r] = cnt;
}

// ---- which: output in range order (as(which, "IntegerRangesList")), then file order -----------
// Per record (bam_which_count_kernel): its (refID, POS + 1) key, the ranges it yields when kept
// and its reference span.  The records a range [s, e] on reference c can overlap -- POS < e and
// POS + span > s - 1 -- are the contiguous run of keys from (c, s - maxspan[c] + 1) to (c, e)
// (bam_which_search_kernel).  The runs are cut into chunks of WHICH_CHUNK records in (range,
// file) order; a count pass, a scan over the chunk counts and a write pass place the pieces, so
// that neither a whole-chromosome range nor one hot range serialises on one CTA.
constexpr int WHICH_ITEMS = 8;
constexpr int WHICH_CHUNK = CTA * WHICH_ITEMS;

struct Which {
    int n;                        // ranges
    const int32_t* ref;           // n: the ranges in output order
    const int32_t* start;
    const int32_t* end;
    const int32_t* ref_off;       // n_ref + 1: the ranges of each reference in the sorted arrays
    const int32_t* s_sorted;      // n: starts, ascending within each reference
    const int32_t* e_sorted;      // n: ends, ascending within each reference
    uint64_t* key;                // records: (refID << 32 | POS + 1); unplaced or malformed: max
    uint32_t* pieces;             // records: ranges a kept record yields, 0 when dropped
    uint32_t* span;               // records: reference span, at least 1 (htslib bam_endpos)
    unsigned int* maxspan;        // n_ref: largest span of a kept record
    unsigned long long* total;    // [0] ranges out [1] chunks
    uint32_t* run_lo;             // n: first record of the range's candidate run
    uint32_t* run_n;              // n: records in the run
    uint32_t* n_chunks;           // n + 1: chunks of the run, scanned into chunk_off
    uint32_t* chunk_off;          // n + 1
};

__device__ __forceinline__ uint64_t rec_key(const uint8_t* p) {
    const int ref = (int)ld_u32(p + 4);
    return ref < 0 ? ~0ull : ((uint64_t)(uint32_t)ref << 32) | (uint64_t)(ld_u32(p + 8) + 1u);
}

// first index in [a, b) whose value is > v
template <class T, class V>
__device__ __forceinline__ int64_t upper_bound_dev(const T* x, int64_t a, int64_t b, V v) {
    while (a < b) {
        const int64_t m = (a + b) >> 1;
        if ((V)x[m] <= v) a = m + 1;
        else b = m;
    }
    return a;
}
template <class T, class V>
__device__ __forceinline__ int64_t lower_bound_dev(const T* x, int64_t a, int64_t b, V v) {
    while (a < b) {
        const int64_t m = (a + b) >> 1;
        if ((V)x[m] < v) a = m + 1;
        else b = m;
    }
    return a;
}

__device__ __forceinline__ bool which_overlaps(uint64_t key, uint32_t span, int64_t s, int64_t e) {
    const int64_t pos0 = (int64_t)(uint32_t)key - 1;
    return pos0 < e && pos0 + (int64_t)span > s - 1;
}

// One thread per record: key, pieces, span, maxspan, the sortedness check over all records, and
// the number of ranges out (pieces x the which ranges the record overlaps, counted by binary
// search in the sorted starts and ends: those with e > POS less those with s > POS + span).
// (__maxnreg__: under __launch_bounds__ alone ptxas settles on 48 registers and spills)
__global__ void __maxnreg__(64)
bam_which_count_kernel(const uint8_t* __restrict__ rec, int64_t n_bytes, const int64_t* __restrict__ off, int64_t n,
                       int n_ref, const int64_t* __restrict__ ref_len, int split, Filter f, Which wh,
                       unsigned int* __restrict__ err) {
    extern __shared__ __align__(16) uint32_t s_tab[];
    stage_tag_table<true>(f, s_tab);
    const int64_t r = (int64_t)blockIdx.x * CTA + threadIdx.x;
    unsigned long long tot = 0;
    int mref = -1;                  // reference of a kept record, for the maxspan update
    unsigned int mspan = 0;
    if (r < n) {
        const int64_t o = off[r], o1 = off[r + 1];
        uint64_t key = ~0ull;
        if (o >= 0 && o1 <= n_bytes && o1 - o >= 36) {
            key = rec_key(rec + o);
            const int64_t op = r > 0 ? off[r - 1] : -1;
            if (op >= 0 && o - op >= 36 && key < rec_key(rec + op)) atomicOr(err, 32u);
        }
        wh.key[r] = key;
        int64_t span = 0;
        const Out none = {nullptr, nullptr, nullptr, nullptr};
        const uint32_t cnt = bam_record<false, true>(rec, n_bytes, o, o1, n_ref, ref_len, split, 0u, none, err, f,
                                                     s_tab, span);
        span = min(max(span, (int64_t)1), (int64_t)1 << 30);
        wh.pieces[r] = cnt;
        wh.span[r] = (uint32_t)span;
        if (cnt) {
            const int ref = (int)(key >> 32);
            const int64_t pos0 = (int64_t)(uint32_t)key - 1;
            mref = ref;
            mspan = (unsigned int)span;
            const int64_t a = wh.ref_off[ref], b = wh.ref_off[ref + 1];
            const int64_t k = (b - upper_bound_dev(wh.e_sorted, a, b, pos0)) -
                              (b - upper_bound_dev(wh.s_sorted, a, b, pos0 + span));
            tot = (unsigned long long)cnt * (unsigned long long)k;
        }
    }
    // sorted records: a warp's kept records share a reference, one atomicMax per reference and warp
    const unsigned int peers = __match_any_sync(0xffffffffu, mref);
    mspan = __reduce_max_sync(peers, mspan);
    if (mref >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicMax(wh.maxspan + mref, mspan);
    for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, d);
    if ((threadIdx.x & 31) == 0 && tot) atomicAdd(wh.total, tot);
}

// One thread per which range: its candidate run of records and the number of chunks of it.
__global__ void __launch_bounds__(CTA)
bam_which_search_kernel(int64_t n, Which wh) {
    const int i = blockIdx.x * CTA + threadIdx.x;
    if (i >= wh.n) return;
    const uint64_t c = (uint64_t)(uint32_t)wh.ref[i] << 32;
    const int64_t s = wh.start[i], e = wh.end[i];
    const int64_t low = max((int64_t)0, s - (int64_t)wh.maxspan[wh.ref[i]] + 1);
    const int64_t lo = lower_bound_dev(wh.key, 0, n, c | (uint64_t)low);
    const int64_t hi = max(lo, upper_bound_dev(wh.key, 0, n, c | (uint64_t)e));    // hi < lo: unsorted records
    const uint32_t nc = (uint32_t)((hi - lo + WHICH_CHUNK - 1) / WHICH_CHUNK);
    wh.run_lo[i] = (uint32_t)lo;
    wh.run_n[i] = (uint32_t)(hi - lo);
    wh.n_chunks[i] = nc;
    if (nc) atomicAdd(wh.total + 1, (unsigned long long)nc);
}

// chunk -> (range, its records [*r0, *r1))
__device__ __forceinline__ int which_chunk(const Which& wh, int64_t c, int64_t* r0, int64_t* r1) {
    const int i = (int)upper_bound_dev(wh.chunk_off, 0, wh.n, (int64_t)c) - 1;
    *r0 = (int64_t)wh.run_lo[i] + (c - (int64_t)wh.chunk_off[i]) * WHICH_CHUNK;
    *r1 = min(*r0 + WHICH_CHUNK, (int64_t)wh.run_lo[i] + wh.run_n[i]);
    return i;
}

// pieces of the records of chunk c that overlap its range; thread t takes WHICH_ITEMS consecutive
// records, so that a block scan of the per-thread counts keeps the file order
__device__ __forceinline__ uint32_t which_thread_pieces(const Which& wh, int i, int64_t r0, int64_t r1) {
    uint32_t v = 0;
    const int64_t s = wh.start[i], e = wh.end[i];
    for (int k = 0; k < WHICH_ITEMS; k++) {
        const int64_t r = r0 + (int64_t)threadIdx.x * WHICH_ITEMS + k;
        if (r < r1 && wh.pieces[r] && which_overlaps(wh.key[r], wh.span[r], s, e)) v += wh.pieces[r];
    }
    return v;
}

__global__ void __launch_bounds__(CTA)
bam_which_chunk_count_kernel(Which wh, uint32_t* __restrict__ chunk_cnt) {
    __shared__ uint32_t wsum[WARPS];
    int64_t r0, r1;
    const int i = which_chunk(wh, blockIdx.x, &r0, &r1);
    uint32_t v = which_thread_pieces(wh, i, r0, r1);
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int k = 0; k < WARPS; k++) t += wsum[k];
        chunk_cnt[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(CTA)
bam_which_write_kernel(const uint8_t* __restrict__ rec, int64_t n_bytes, const int64_t* __restrict__ off, int n_ref,
                       const int64_t* __restrict__ ref_len, int split, Which wh,
                       const uint32_t* __restrict__ chunk_base, Out out, unsigned int* __restrict__ err) {
    __shared__ uint32_t wsum[WARPS];
    int64_t r0, r1;
    const int i = which_chunk(wh, blockIdx.x, &r0, &r1);
    const uint32_t v = which_thread_pieces(wh, i, r0, r1);
    const int lane = threadIdx.x & 31;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    uint32_t w = chunk_base[blockIdx.x] + inc - v;
    for (int k = 0; k < (int)(threadIdx.x >> 5); k++) w += wsum[k];
    if (v == 0) return;
    const int64_t s = wh.start[i], e = wh.end[i];
    const Filter none = {};
    for (int k = 0; k < WHICH_ITEMS; k++) {
        const int64_t r = r0 + (int64_t)threadIdx.x * WHICH_ITEMS + k;
        if (r < r1 && wh.pieces[r] && which_overlaps(wh.key[r], wh.span[r], s, e)) {
            int64_t span;
            // the record passed the filters in the count pass: the plain walk writes its pieces
            w += bam_record<true, false>(rec, n_bytes, off[r], off[r + 1], n_ref, ref_len, split, w, out, err, none,
                                         nullptr, span);
        }
    }
}

// ------------------------------------------------------------------------------- BED ----------
__device__ __forceinline__ int nl_count16(uint4 v, int valid) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    int c = 0;
#pragma unroll
    for (int k = 0; k < 16; k++)
        if (k < valid && ((w[k >> 2] >> ((k & 3) * 8)) & 0xffu) == (uint32_t)'\n') c++;
    return c;
}

// thread i looks at the bytes [16 i, 16 i + 16); block totals of the newline count
__global__ void __launch_bounds__(CTA)
bed_nl_count_kernel(const uint4* __restrict__ text, int64_t n_bytes, uint32_t* __restrict__ block_cnt) {
    __shared__ int wsum[WARPS];
    const int64_t i = (int64_t)blockIdx.x * CTA + threadIdx.x;
    const int64_t lo = i * 16;
    int c = 0;
    if (lo < n_bytes) c = nl_count16(__ldg(text + i), (int)min((int64_t)16, n_bytes - lo));
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int k = 0; k < WARPS; k++) t += wsum[k];
        block_cnt[blockIdx.x] = (uint32_t)t;
    }
}

// starts[0] = 0, starts[k] = position after the k-th newline
__global__ void __launch_bounds__(CTA)
bed_nl_write_kernel(const uint4* __restrict__ text, int64_t n_bytes, const uint32_t* __restrict__ block_base,
                    int64_t* __restrict__ starts) {
    __shared__ int wsum[WARPS];
    const int64_t i = (int64_t)blockIdx.x * CTA + threadIdx.x;
    const int64_t lo = i * 16;
    const int valid = lo < n_bytes ? (int)min((int64_t)16, n_bytes - lo) : 0;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (valid) v = __ldg(text + i);
    const int c = nl_count16(v, valid);
    const int lane = threadIdx.x & 31;
    int inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    int base = inc - c;
    for (int k = 0; k < (int)(threadIdx.x >> 5); k++) base += wsum[k];
    int64_t at = (int64_t)block_base[blockIdx.x] + base + 1;
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 16; k++)
        if (k < valid && ((w[k >> 2] >> ((k & 3) * 8)) & 0xffu) == (uint32_t)'\n') starts[at++] = lo + k + 1;
    if (i == 0) starts[0] = 0;
}

struct NameTable {
    const char* blob;        // the names, sorted, one after the other
    const int32_t* name_off; // n + 1
    const int32_t* id;       // seqlevel index of the sorted name
    int n;
};

__device__ __forceinline__ bool is_sep(uint8_t c) { return c == '\t' || c == ' '; }

__device__ __forceinline__ int name_cmp(const uint8_t* a, int la, const char* b, int lb) {
    const int m = min(la, lb);
    for (int k = 0; k < m; k++) {
        const int d = (int)a[k] - (int)(uint8_t)b[k];
        if (d) return d;
    }
    return la - lb;
}

// err bits: 1 chromosome name not among the seqlevels, 2 a data line with fewer than three
//           fields or a bad number, 4 a strand field other than + - . *
// One thread per line.  Skipped: empty lines, comments (#), "track" and "browser" lines.
template <bool WRITE>
__global__ void __launch_bounds__(CTA)
bed_lines_kernel(const uint8_t* __restrict__ text, int64_t n_bytes, const int64_t* __restrict__ starts,
                 int64_t n_nl, int64_t n_lines, NameTable names, uint32_t* __restrict__ counts,
                 const uint32_t* __restrict__ where, Out out, unsigned int* __restrict__ err) {
    const int64_t j = (int64_t)blockIdx.x * CTA + threadIdx.x;
    if (j >= n_lines) return;
    int64_t a = starts[j], b = j < n_nl ? starts[j + 1] - 1 : n_bytes;
    if (b > a && text[b - 1] == '\r') b--;
    while (a < b && is_sep(text[a])) a++;
    uint32_t cnt = 0;
    do {
        if (a >= b || text[a] == '#') break;
        int64_t f0 = a, f1 = a;
        while (f1 < b && !is_sep(text[f1])) f1++;
        const int l0 = (int)(f1 - f0);
        if ((l0 == 5 && name_cmp(text + f0, 5, "track", 5) == 0) ||
            (l0 == 7 && name_cmp(text + f0, 7, "browser", 7) == 0))
            break;
        int lo = 0, hi = names.n - 1, found = -1;
        while (lo <= hi) {
            const int mid = (lo + hi) >> 1;
            const int c = name_cmp(text + f0, l0, names.blob + names.name_off[mid],
                                   names.name_off[mid + 1] - names.name_off[mid]);
            if (c == 0) {
                found = mid;
                break;
            }
            if (c < 0) hi = mid - 1;
            else lo = mid + 1;
        }
        if (found < 0) {
            atomicOr(err, 1u);
            break;
        }
        int64_t num[2] = {0, 0};
        bool bad = false;
        int64_t q = f1;
        for (int f = 0; f < 2; f++) {
            while (q < b && is_sep(text[q])) q++;
            const int64_t q0 = q;
            int64_t v = 0;
            while (q < b && !is_sep(text[q])) {
                const int dgt = (int)text[q] - '0';
                if (dgt < 0 || dgt > 9 || v > 0x7fffffff) bad = true;
                v = v * 10 + dgt;
                q++;
            }
            if (q == q0 || v > 0x7ffffffe) bad = true;
            num[f] = v;
        }
        if (bad) {
            atomicOr(err, 2u);
            break;
        }
        int8_t st = 0;
        for (int f = 3; f <= 5; f++) {              // name, score, strand
            while (q < b && is_sep(text[q])) q++;
            const int64_t q0 = q;
            while (q < b && !is_sep(text[q])) q++;
            if (f == 5 && q > q0) {
                const uint8_t c = text[q0];
                if (q - q0 != 1 || !(c == '+' || c == '-' || c == '.' || c == '*')) atomicOr(err, 4u);
                st = c == '+' ? 1 : (c == '-' ? -1 : 0);
            }
        }
        if (WRITE) {
            const uint32_t w = where[j];
            out.chrom[w] = names.id[found];
            out.start[w] = (int32_t)(num[0] + 1);   // BED starts are 0-based, ends exclusive
            out.end[w] = (int32_t)num[1];
            out.strand[w] = st;
        }
        cnt = 1;
    } while (false);
    if (!WRITE) counts[j] = cnt;
}

int new_decoded(Decoded** d, int* h) {
    *h = g_next_decoded++;
    g_decoded[*h] = std::unique_ptr<Decoded>(new Decoded());
    *d = g_decoded[*h].get();
    return RCP_OK;
}

int alloc_out(Decoded& d, int64_t n) {
    d.n = n;
    RCP_TRY(dalloc(&d.chrom, (size_t)n));
    RCP_TRY(dalloc(&d.start, (size_t)n));
    RCP_TRY(dalloc(&d.end, (size_t)n));
    RCP_TRY(dalloc(&d.strand, (size_t)n));
    return RCP_OK;
}

int bam_check_args(const char* fn, const uint8_t* rec, int64_t n_bytes, const int64_t* offsets, int64_t n_records,
                   int n_ref, const int64_t* ref_len, int mem, const int* decoded_out, const int64_t* n_out) {
    RCP_TRY(require_ready());
    if (n_bytes < 0 || n_records < 0 || n_ref < 0 || decoded_out == nullptr || n_out == nullptr ||
        (n_records > 0 && (rec == nullptr || offsets == nullptr)) || (n_ref > 0 && ref_len == nullptr))
        return fail(RCP_ERR_ARG, "%s: bad argument", fn);
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    if (n_records >= 0x7ffffff0ll) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31 - 17 alignment records");
    return RCP_OK;
}

int bam_errors(unsigned int h_err, int n_ref) {
    if (h_err & 1u) return fail(RCP_ERR_DATA, "BAM records: the offsets do not follow the record chain, or a record is truncated");
    if (h_err & 2u) return fail(RCP_ERR_DATA, "BAM records: a refID is outside the header's %d references", n_ref);
    if (h_err & 4u) return fail(RCP_ERR_DATA, "BAM records: a CIGAR operation code is above 8");
    if (h_err & 8u) return fail(RCP_ERR_DATA, "BAM records: a mapped record has no CIGAR (GAlignments needs one)");
    if (h_err & 16u) return fail(RCP_ERR_DATA, "BAM records: an aux field runs past its record or has an unknown type");
    if (h_err & 32u)
        return fail(RCP_ERR_DATA, "BAM records: `which` needs records sorted by (refID, POS), unplaced ones last");
    return RCP_OK;
}

// A new decoded handle of n ranges; write(out) queues the kernel that fills it.
template <class F>
int bam_output(int64_t n, int* decoded_out, int64_t* n_out, F write) {
    Decoded* d;
    int h;
    RCP_TRY(new_decoded(&d, &h));
    int rc = alloc_out(*d, n);
    if (rc == RCP_OK && n > 0) rc = write(Out{d->chrom, d->start, d->end, d->strand});
    if (rc != RCP_OK) {
        decoded_release(*d);
        g_decoded.erase(h);
        return rc;
    }
    *decoded_out = h;
    *n_out = n;
    return RCP_OK;
}

// count -> exclusive scan -> write: the ranges in file order
template <bool FILTER>
int bam_decode_file_order(const uint8_t* rec, int64_t n_bytes, const int64_t* off, int64_t n_records, int n_ref,
                          const int64_t* ref_len, int split, const Filter& f, int* decoded_out, int64_t* n_out) {
    Arena A;
    const size_t n = (size_t)n_records, smem = (size_t)f.table_words * 4;
    RCP_TRY(A.reserve(Arena::pad(16) + Arena::pad((n + 1) * 4) * 2));
    unsigned int* err = A.take<unsigned int>(4);        // [0] err [1] total
    uint32_t* counts = A.take<uint32_t>(n + 1);
    uint32_t* where = A.take<uint32_t>(n + 1);
    RCP_CUDA(cudaMemsetAsync(err, 0, 16, g_ctx.stream));
    const Out none = {nullptr, nullptr, nullptr, nullptr};
    if (n_records > 0) {
        bam_records_kernel<false, FILTER><<<blocks_for(n_records, CTA), CTA, smem, g_ctx.stream>>>(
            rec, n_bytes, off, n_records, n_ref, ref_len, split, counts, nullptr, none, err, f);
        RCP_LAUNCHED();
        RCP_TRY(exclusive_scan_u32(counts, where, n_records, err + 1));
    }
    unsigned int h_err = 0, h_total = 0;
    FetchItem items[2] = {{err, &h_err, 4}, {err + 1, &h_total, 4}};
    RCP_TRY(fetch_and_sync(items, 2));
    RCP_TRY(bam_errors(h_err, n_ref));
    return bam_output((int64_t)h_total, decoded_out, n_out, [&](Out out) -> int {
        bam_records_kernel<true, FILTER><<<blocks_for(n_records, CTA), CTA, smem, g_ctx.stream>>>(
            rec, n_bytes, off, n_records, n_ref, ref_len, split, nullptr, where, out, err, f);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess) return fail(RCP_ERR_CUDA, "bam_records_kernel launch failed");
        return RCP_OK;
    });
}

// which: the records of every range in range order, then file order
int bam_decode_which(const uint8_t* rec, int64_t n_bytes, const int64_t* off, int64_t n_records, int n_ref,
                     const int64_t* ref_len, int split, const Filter& f, const std::vector<int32_t>& wtab, int n_which,
                     int* decoded_out, int64_t* n_out) {
    const size_t n = (size_t)n_records, W = (size_t)n_which, smem = (size_t)f.table_words * 4;
    Arena A;
    RCP_TRY(A.reserve(Arena::pad(32) + Arena::pad(wtab.size() * 4) + Arena::pad(std::max(n, (size_t)1) * 8) +
                      Arena::pad(std::max(n, (size_t)1) * 4) * 2 + Arena::pad((size_t)std::max(n_ref, 1) * 4) +
                      Arena::pad(W * 4) * 2 + Arena::pad((W + 1) * 4) * 2));
    unsigned long long* stat = A.take<unsigned long long>(4);   // [0] ranges out [1] chunks [2] err
    unsigned int* err = reinterpret_cast<unsigned int*>(stat + 2);
    int32_t* d_wtab = A.take<int32_t>(wtab.size());
    Which wh;
    wh.n = n_which;
    wh.ref = d_wtab;
    wh.start = d_wtab + W;
    wh.end = d_wtab + 2 * W;
    wh.s_sorted = d_wtab + 3 * W;
    wh.e_sorted = d_wtab + 4 * W;
    wh.ref_off = d_wtab + 5 * W;
    wh.key = A.take<uint64_t>(std::max(n, (size_t)1));
    wh.pieces = A.take<uint32_t>(std::max(n, (size_t)1));
    wh.span = A.take<uint32_t>(std::max(n, (size_t)1));
    wh.maxspan = A.take<unsigned int>((size_t)std::max(n_ref, 1));
    wh.total = stat;
    wh.run_lo = A.take<uint32_t>(W);
    wh.run_n = A.take<uint32_t>(W);
    wh.n_chunks = A.take<uint32_t>(W + 1);
    wh.chunk_off = A.take<uint32_t>(W + 1);
    RCP_CUDA(cudaMemsetAsync(stat, 0, 32, g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(wh.maxspan, 0, (size_t)std::max(n_ref, 1) * 4, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_wtab, wtab.data(), wtab.size() * 4, cudaMemcpyHostToDevice, g_ctx.stream));
    if (n_records > 0) {
        bam_which_count_kernel<<<blocks_for(n_records, CTA), CTA, smem, g_ctx.stream>>>(
            rec, n_bytes, off, n_records, n_ref, ref_len, split, f, wh, err);
        RCP_LAUNCHED();
        bam_which_search_kernel<<<blocks_for(n_which, CTA), CTA, 0, g_ctx.stream>>>(n_records, wh);
        RCP_LAUNCHED();
        RCP_TRY(exclusive_scan_u32(wh.n_chunks, wh.chunk_off, n_which, nullptr));
    }
    unsigned long long h_stat[3] = {0, 0, 0};
    FetchItem items[1] = {{stat, h_stat, 24}};
    RCP_TRY(fetch_and_sync(items, 1));
    RCP_TRY(bam_errors((unsigned int)h_stat[2], n_ref));
    if (h_stat[0] >= 0x7ffffff0ull || h_stat[1] >= 0x7ffffff0ull)
        return fail(RCP_ERR_UNSUPPORTED, "which: more than 2^31 - 17 ranges out or record chunks");
    const int64_t n_chunks = (int64_t)h_stat[1];
    return bam_output((int64_t)h_stat[0], decoded_out, n_out, [&](Out out) -> int {
        Arena B;
        RCP_TRY(B.reserve(Arena::pad((size_t)n_chunks * 4) * 2));
        uint32_t* chunk_cnt = B.take<uint32_t>((size_t)n_chunks);
        uint32_t* chunk_base = B.take<uint32_t>((size_t)n_chunks);
        bam_which_chunk_count_kernel<<<(unsigned)n_chunks, CTA, 0, g_ctx.stream>>>(wh, chunk_cnt);
        RCP_LAUNCHED();
        RCP_TRY(exclusive_scan_u32(chunk_cnt, chunk_base, n_chunks, nullptr));
        bam_which_write_kernel<<<(unsigned)n_chunks, CTA, 0, g_ctx.stream>>>(rec, n_bytes, off, n_ref, ref_len, split,
                                                                             wh, chunk_base, out, err);
        RCP_LAUNCHED();
        return RCP_OK;
    });
}

}  // namespace

void decoded_release_all() {
    for (auto& kv : g_decoded) decoded_release(*kv.second);
    g_decoded.clear();
}

}  // namespace rcp

using namespace rcp;

extern "C" {

int rcp_bam_index(const uint8_t* rec, int64_t n_bytes, int64_t* n_records_out, int64_t* offsets_out,
                  int64_t capacity) {
    if (n_bytes < 0 || (n_bytes > 0 && rec == nullptr) || n_records_out == nullptr)
        return fail(RCP_ERR_ARG, "rcp_bam_index: bad argument");
    int64_t p = 0, n = 0;
    while (p < n_bytes) {
        if (n_bytes - p < 4) return fail(RCP_ERR_DATA, "BAM records: truncated block_size at byte %lld", (long long)p);
        int32_t bs;
        memcpy(&bs, rec + p, 4);
        if (bs < 32 || (int64_t)bs + 4 > n_bytes - p)
            return fail(RCP_ERR_DATA, "BAM records: record %lld at byte %lld has block_size %d", (long long)n,
                        (long long)p, (int)bs);
        if (offsets_out) {
            if (n + 1 >= capacity)      // room for this record's offset and for the end
                return fail(RCP_ERR_ARG, "rcp_bam_index: offsets_out has %lld entries, the file more records", (long long)capacity);
            offsets_out[n] = p;
        }
        p += 4 + (int64_t)bs;
        n++;
    }
    if (offsets_out) {
        if (capacity < 1) return fail(RCP_ERR_ARG, "rcp_bam_index: offsets_out needs records + 1 entries");
        offsets_out[n] = p;
    }
    *n_records_out = n;
    return RCP_OK;
}

int rcp_bam_decode(const uint8_t* rec, int64_t n_bytes, const int64_t* offsets, int64_t n_records, int n_ref,
                   const int64_t* ref_len, int splice_split, int mem, int* decoded_out, int64_t* n_out) {
    RCP_TRY(bam_check_args("rcp_bam_decode", rec, n_bytes, offsets, n_records, n_ref, ref_len, mem, decoded_out, n_out));
    DevIn<uint8_t> d_rec;
    DevIn<int64_t> d_off, d_len;
    RCP_TRY(d_rec.init(rec, (size_t)n_bytes, mem));
    RCP_TRY(d_off.init(offsets, (size_t)n_records + 1, mem));
    RCP_TRY(d_len.init(ref_len, (size_t)std::max(n_ref, 1), RCP_MEM_HOST));
    return bam_decode_file_order<false>(d_rec.ptr, n_bytes, d_off.ptr, n_records, n_ref, d_len.ptr,
                                        splice_split ? 1 : 0, Filter{}, decoded_out, n_out);
}

int rcp_bam_decode_param(const uint8_t* rec, int64_t n_bytes, const int64_t* offsets, int64_t n_records, int n_ref,
                         const int64_t* ref_len, int splice_split, int mem, const int32_t* flag, int mapq_min,
                         int simple_cigar, int n_which, const int32_t* which_ref, const int32_t* which_start,
                         const int32_t* which_end, int n_tags, const char* tag_names, const int32_t* tag_ptr,
                         const int32_t* tag_type, const int64_t* int_values, const char* const* str_values,
                         int* decoded_out, int64_t* n_out) {
    RCP_TRY(bam_check_args("rcp_bam_decode_param", rec, n_bytes, offsets, n_records, n_ref, ref_len, mem,
                           decoded_out, n_out));
    Filter f = {};
    f.keep0 = flag ? (uint32_t)flag[0] : 0xfffu;
    f.keep1 = flag ? (uint32_t)flag[1] : 0xfffu;
    f.mapq_min = mapq_min;
    f.simple_cigar = simple_cigar ? 1 : 0;
    // the tag table (see Filter)
    if (n_tags < 0 || n_tags > 32) return fail(RCP_ERR_UNSUPPORTED, "tagFilter: %d tags (at most 32)", n_tags);
    if (n_tags > 0 && (tag_names == nullptr || tag_ptr == nullptr || tag_type == nullptr))
        return fail(RCP_ERR_ARG, "rcp_bam_decode_param: bad tag filter");
    std::vector<Tag> tags((size_t)n_tags);
    std::vector<int64_t> ival;
    std::vector<uint32_t> soff(1, 0);
    std::string sbytes;
    for (int k = 0; k < n_tags; k++) {
        const int32_t a = tag_ptr[k], b = tag_ptr[k + 1];
        if (a < 0 || b < a || (k == 0 && a != 0) || (tag_type[k] != 0 && tag_type[k] != 1))
            return fail(RCP_ERR_ARG, "rcp_bam_decode_param: bad tag filter (tag %d)", k);
        Tag& t = tags[(size_t)k];
        t.name = (uint32_t)(uint8_t)tag_names[2 * k] | ((uint32_t)(uint8_t)tag_names[2 * k + 1] << 8);
        t.is_str = (uint32_t)tag_type[k];
        if (t.is_str) {
            t.v0 = (uint32_t)(soff.size() - 1);
            for (int32_t j = a; j < b; j++) {
                if (str_values == nullptr || str_values[j] == nullptr)
                    return fail(RCP_ERR_ARG, "rcp_bam_decode_param: tag %d: NULL string value", k);
                sbytes += str_values[j];
                soff.push_back((uint32_t)sbytes.size());
            }
            t.v1 = (uint32_t)(soff.size() - 1);
        } else {
            if (b > a && int_values == nullptr) return fail(RCP_ERR_ARG, "rcp_bam_decode_param: int_values is NULL");
            t.v0 = (uint32_t)ival.size();
            for (int32_t j = a; j < b; j++) ival.push_back(int_values[j]);
            t.v1 = (uint32_t)ival.size();
        }
    }
    std::vector<uint32_t> table;
    if (n_tags > 0) {
        const size_t w_tags = 4 * (size_t)n_tags, w_int = 2 * ival.size(), w_str = soff.size() + (sbytes.size() + 3) / 4;
        if ((w_tags + w_int + w_str) * 4 > 32768)
            return fail(RCP_ERR_UNSUPPORTED, "tagFilter: the filter values take more than 32 KB");
        table.assign(w_tags + w_int + w_str, 0u);
        memcpy(table.data(), tags.data(), w_tags * 4);
        memcpy(table.data() + w_tags, ival.data(), w_int * 4);
        memcpy(table.data() + w_tags + w_int, soff.data(), soff.size() * 4);
        memcpy(table.data() + w_tags + w_int + soff.size(), sbytes.data(), sbytes.size());
        f.n_tags = n_tags;
        f.n_int = (int)ival.size();
        f.n_str = (int)soff.size() - 1;
        f.table_words = (int)table.size();
    }
    // which: the ranges in output order, then per reference their starts and their ends sorted
    if (n_which < 0 || (n_which > 0 && (which_ref == nullptr || which_start == nullptr || which_end == nullptr)))
        return fail(RCP_ERR_ARG, "rcp_bam_decode_param: bad which ranges");
    const size_t W = (size_t)n_which;
    std::vector<int32_t> wtab;
    if (n_which > 0) {
        wtab.assign(5 * W + (size_t)n_ref + 1, 0);
        std::vector<int32_t> cnt((size_t)n_ref + 1, 0);
        for (size_t i = 0; i < W; i++) {
            const int32_t c = which_ref[i], s = which_start[i], e = which_end[i];
            if (c < 0 || c >= n_ref)
                return fail(RCP_ERR_ARG, "which: range %zu is on reference %d, the header has %d", i, (int)c, n_ref);
            if (s < 1 || e < s || e > 536870912)
                return fail(RCP_ERR_ARG, "which: range %zu [%d, %d] needs 1 <= start <= end <= 536870912", i, (int)s,
                            (int)e);
            wtab[i] = c;
            wtab[W + i] = s;
            wtab[2 * W + i] = e;
            cnt[(size_t)c + 1]++;
        }
        int32_t* ref_off = wtab.data() + 5 * W;
        for (int c = 0; c < n_ref; c++) ref_off[c + 1] = ref_off[c] + cnt[(size_t)c + 1];
        std::vector<int32_t> fill(ref_off, ref_off + n_ref);
        for (size_t i = 0; i < W; i++) {
            const int32_t at = fill[(size_t)wtab[i]]++;
            wtab[3 * W + (size_t)at] = wtab[W + i];
            wtab[4 * W + (size_t)at] = wtab[2 * W + i];
        }
        for (int c = 0; c < n_ref; c++) {
            std::sort(wtab.begin() + 3 * W + ref_off[c], wtab.begin() + 3 * W + ref_off[c + 1]);
            std::sort(wtab.begin() + 4 * W + ref_off[c], wtab.begin() + 4 * W + ref_off[c + 1]);
        }
    }
    DevIn<uint8_t> d_rec;
    DevIn<int64_t> d_off, d_len;
    DevIn<uint32_t> d_table;
    RCP_TRY(d_rec.init(rec, (size_t)n_bytes, mem));
    RCP_TRY(d_off.init(offsets, (size_t)n_records + 1, mem));
    RCP_TRY(d_len.init(ref_len, (size_t)std::max(n_ref, 1), RCP_MEM_HOST));
    RCP_TRY(d_table.init(table.empty() ? nullptr : table.data(), table.size(), RCP_MEM_HOST));
    f.table = d_table.ptr;
    const int split = splice_split ? 1 : 0;
    if (n_which == 0)
        return bam_decode_file_order<true>(d_rec.ptr, n_bytes, d_off.ptr, n_records, n_ref, d_len.ptr, split, f,
                                           decoded_out, n_out);
    return bam_decode_which(d_rec.ptr, n_bytes, d_off.ptr, n_records, n_ref, d_len.ptr, split, f, wtab, n_which,
                            decoded_out, n_out);
}

int rcp_bed_decode(const char* text, int64_t n_bytes, int n_names, const char* const* names, int mem,
                   int* decoded_out, int64_t* n_out) {
    RCP_TRY(require_ready());
    if (n_bytes < 0 || (n_bytes > 0 && text == nullptr) || n_names < 1 || names == nullptr ||
        decoded_out == nullptr || n_out == nullptr)
        return fail(RCP_ERR_ARG, "rcp_bed_decode: bad argument");
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    // the seqlevels, sorted by name for the device's binary search
    std::vector<int32_t> order((size_t)n_names);
    for (int i = 0; i < n_names; i++) {
        if (names[i] == nullptr) return fail(RCP_ERR_ARG, "rcp_bed_decode: names[%d] is NULL", i);
        order[(size_t)i] = i;
    }
    std::sort(order.begin(), order.end(), [&](int32_t x, int32_t y) {
        const size_t lx = strlen(names[x]), ly = strlen(names[y]);
        const int c = memcmp(names[x], names[y], std::min(lx, ly));
        return c != 0 ? c < 0 : lx < ly;
    });
    std::string blob;
    std::vector<int32_t> noff((size_t)n_names + 1);
    for (int i = 0; i < n_names; i++) {
        noff[(size_t)i] = (int32_t)blob.size();
        blob += names[order[(size_t)i]];
        if (i > 0 && blob.compare((size_t)noff[(size_t)i - 1], (size_t)(noff[(size_t)i] - noff[(size_t)i - 1]),
                                  names[order[(size_t)i]]) == 0)
            return fail(RCP_ERR_ARG, "rcp_bed_decode: seqlevel '%s' appears twice", names[order[(size_t)i]]);
    }
    noff[(size_t)n_names] = (int32_t)blob.size();
    // the text, 16-byte aligned with 16 readable bytes past the end (our own copy unless the
    // caller's device pointer is aligned; the tail of the last vector is masked by n_bytes)
    const size_t padded = ((size_t)n_bytes + 15) / 16 * 16 + 16;
    uint8_t* d_text = nullptr;
    RCP_TRY(dalloc(&d_text, padded));
    struct Free {
        uint8_t*& p;
        ~Free() { dfree(p); }
    } free_text{d_text};
    if (n_bytes > 0)
        RCP_CUDA(cudaMemcpyAsync(d_text, text, (size_t)n_bytes,
                                 mem == RCP_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, g_ctx.stream));
    const int64_t n_vec = (n_bytes + 15) / 16;
    const unsigned blocks = std::max(1u, blocks_for(n_vec, CTA));
    Arena A;
    RCP_TRY(A.reserve(Arena::pad(16) + Arena::pad(((size_t)blocks + 1) * 4) * 2 + Arena::pad(blob.size() + 1) +
                      Arena::pad(((size_t)n_names + 1) * 4) * 2));
    unsigned int* err = A.take<unsigned int>(4);        // [0] err [1] newlines [2] lines kept
    uint32_t* bcnt = A.take<uint32_t>((size_t)blocks + 1);
    uint32_t* bbase = A.take<uint32_t>((size_t)blocks + 1);
    char* d_blob = A.take<char>(blob.size() + 1);
    int32_t* d_noff = A.take<int32_t>((size_t)n_names + 1);
    int32_t* d_id = A.take<int32_t>((size_t)n_names + 1);
    RCP_CUDA(cudaMemsetAsync(err, 0, 16, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_noff, noff.data(), noff.size() * 4, cudaMemcpyHostToDevice, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(d_id, order.data(), order.size() * 4, cudaMemcpyHostToDevice, g_ctx.stream));
    bed_nl_count_kernel<<<blocks, CTA, 0, g_ctx.stream>>>(reinterpret_cast<const uint4*>(d_text), n_bytes, bcnt);
    RCP_LAUNCHED();
    RCP_TRY(exclusive_scan_u32(bcnt, bbase, (int64_t)blocks, err + 1));
    unsigned int h_nl = 0;
    uint8_t last = '\n';
    {
        FetchItem it[1] = {{err + 1, &h_nl, 4}};
        RCP_TRY(fetch_and_sync(it, 1));
        if (n_bytes > 0) {
            RCP_CUDA(cudaMemcpyAsync(&last, d_text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, g_ctx.stream));
            RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        }
    }
    const int64_t n_nl = (int64_t)h_nl, n_lines = n_nl + ((n_bytes > 0 && last != '\n') ? 1 : 0);
    if (n_lines >= 0x7ffffff0ll) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31 - 17 lines");
    Arena B;
    RCP_TRY(B.reserve(Arena::pad(((size_t)n_nl + 2) * 8) + Arena::pad(((size_t)n_lines + 1) * 4) * 2));
    int64_t* starts = B.take<int64_t>((size_t)n_nl + 2);
    uint32_t* counts = B.take<uint32_t>((size_t)n_lines + 1);
    uint32_t* where = B.take<uint32_t>((size_t)n_lines + 1);
    bed_nl_write_kernel<<<blocks, CTA, 0, g_ctx.stream>>>(reinterpret_cast<const uint4*>(d_text), n_bytes, bbase, starts);
    RCP_LAUNCHED();
    const NameTable nt = {d_blob, d_noff, d_id, n_names};
    const Out none = {nullptr, nullptr, nullptr, nullptr};
    if (n_lines > 0) {
        bed_lines_kernel<false><<<blocks_for(n_lines, CTA), CTA, 0, g_ctx.stream>>>(d_text, n_bytes, starts, n_nl, n_lines,
                                                                                  nt, counts, nullptr, none, err);
        RCP_LAUNCHED();
        RCP_TRY(exclusive_scan_u32(counts, where, n_lines, err + 2));
    }
    unsigned int h_err = 0, h_total = 0;
    FetchItem items[2] = {{err, &h_err, 4}, {err + 2, &h_total, 4}};
    RCP_TRY(fetch_and_sync(items, 2));
    if (h_err & 1u) return fail(RCP_ERR_DATA, "BED: a chromosome name is not among the %d seqlevels", n_names);
    if (h_err & 2u) return fail(RCP_ERR_DATA, "BED: a data line has fewer than three fields or a bad coordinate");
    if (h_err & 4u) return fail(RCP_ERR_DATA, "BED: a strand field is not one of + - . *");
    Decoded* d;
    int h;
    RCP_TRY(new_decoded(&d, &h));
    int rc = alloc_out(*d, (int64_t)h_total);
    if (rc == RCP_OK && n_lines > 0) {
        const Out out = {d->chrom, d->start, d->end, d->strand};
        bed_lines_kernel<true><<<blocks_for(n_lines, CTA), CTA, 0, g_ctx.stream>>>(d_text, n_bytes, starts, n_nl, n_lines, nt,
                                                                                 nullptr, where, out, err);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess) rc = fail(RCP_ERR_CUDA, "bed_lines_kernel launch failed");
    }
    if (rc != RCP_OK) {
        decoded_release(*d);
        g_decoded.erase(h);
        return rc;
    }
    *decoded_out = h;
    *n_out = (int64_t)h_total;
    return RCP_OK;
}

int rcp_decoded_fetch(int decoded, int32_t* chrom, int32_t* start, int32_t* end, int8_t* strand, int64_t capacity) {
    RCP_TRY(require_ready());
    auto it = g_decoded.find(decoded);
    if (it == g_decoded.end()) return fail(RCP_ERR_HANDLE, "unknown decoded handle %d", decoded);
    const Decoded& d = *it->second;
    if (capacity < d.n) return fail(RCP_ERR_ARG, "rcp_decoded_fetch: capacity %lld < %lld ranges", (long long)capacity, (long long)d.n);
    const size_t n = (size_t)d.n;
    if (n == 0) return RCP_OK;
    if (chrom) RCP_CUDA(cudaMemcpyAsync(chrom, d.chrom, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (start) RCP_CUDA(cudaMemcpyAsync(start, d.start, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (end) RCP_CUDA(cudaMemcpyAsync(end, d.end, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (strand) RCP_CUDA(cudaMemcpyAsync(strand, d.strand, n, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return RCP_OK;
}

int rcp_decoded_free(int decoded) {
    auto it = g_decoded.find(decoded);
    if (it == g_decoded.end()) return fail(RCP_ERR_HANDLE, "unknown decoded handle %d", decoded);
    decoded_release(*it->second);
    g_decoded.erase(it);
    return RCP_OK;
}

int rcp_reads_load_decoded(int decoded, int n_chrom, const int64_t* chrom_len, int frag_len, int* reads_out) {
    RCP_TRY(require_ready());
    auto it = g_decoded.find(decoded);
    if (it == g_decoded.end()) return fail(RCP_ERR_HANDLE, "unknown decoded handle %d", decoded);
    const Decoded& d = *it->second;
    return rcp_reads_load(d.n, d.chrom, d.start, d.end, d.strand, n_chrom, chrom_len, frag_len, RCP_MEM_DEVICE,
                          reads_out);
}

int rcp_decoded_width_quantile(int decoded, double prob, double* quantile_out, int64_t* n_le_out) {
    RCP_TRY(require_ready());
    auto it = g_decoded.find(decoded);
    if (it == g_decoded.end()) return fail(RCP_ERR_HANDLE, "unknown decoded handle %d", decoded);
    const Decoded& d = *it->second;
    return rcp_reads_width_quantile(d.n, d.start, d.end, prob, RCP_MEM_DEVICE, quantile_out, n_le_out);
}

int rcp_reads_load_decoded_select(int decoded, double max_width, int64_t k, const int32_t* idx, int n_chrom,
                                  const int64_t* chrom_len, int frag_len, int64_t* n_kept_out, int* reads_out) {
    RCP_TRY(require_ready());
    auto it = g_decoded.find(decoded);
    if (it == g_decoded.end()) return fail(RCP_ERR_HANDLE, "unknown decoded handle %d", decoded);
    if (k < 0 || (k > 0 && idx == nullptr)) return fail(RCP_ERR_ARG, "rcp_reads_load_decoded_select: bad index");
    const Decoded& d = *it->second;
    DevIn<int32_t> d_idx;
    RCP_TRY(d_idx.init(idx, (size_t)k, RCP_MEM_HOST));
    return rcp_reads_load_select(d.n, d.chrom, d.start, d.end, d.strand, max_width, k, d_idx.ptr, n_chrom, chrom_len,
                                 frag_len, RCP_MEM_DEVICE, n_kept_out, reads_out);
}

}  // extern "C"
