// BigWig input (coverageFromBigWig of the reference, /root/reference/R/coverage.R:228-322, which
// reads `import.bw(file, as = "RleList")` and subscripts each chromosome's numeric vector by the
// window like the reads path).
//
// Load (rcp_bigwig_load): the UCSC bbi container (Kent et al. 2010; the layouts of bbiFile.h /
// bwgInternal.h) is parsed on the host -- 64-byte header, the chromosome B+ tree, the leaves of
// the R-tree index that locate the data blocks -- and the blocks are inflated by the host thread
// pool of bgzf.cu (zlib streams, or copied when the file is stored uncompressed).  The inflated
// sections cross PCIe once and are expanded on the device into SoA items (start, end 1-based
// closed, float value), validated there, with one host synchronisation for the verdict.
//
// Coverage (rcp_signal_coverage): every range of the mask is cut into warp tiles of ST positions.
// A warp finds the first item of its tile by one binary search over the chromosome's item ends
// (items are sorted and disjoint), paints the items into a shared-memory tile (zeros between
// them), then stores the tile coalesced -- mirrored on '-' elements.  The item spans are
// disjoint, so no atomics are needed.  The result is an ordinary coverage handle (DESIGN.md §3
// layout: offsets multiples of 32 words, len = 0 for NULL) whose words hold float bits.
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "cov_common.cuh"
#include "rcp_internal.cuh"

namespace rcp {
namespace {

using covk::blocks_for;

constexpr uint32_t BIGWIG_MAGIC = 0x888FFC26u;
constexpr uint32_t BIGBED_MAGIC = 0x8789F2EBu;
constexpr uint32_t CHROM_TREE_MAGIC = 0x78CA8C91u;
constexpr uint32_t RTREE_MAGIC = 0x2468ACE0u;
constexpr int SECTION_HEAD = 24;

struct Signal {
    int n_chrom = 0;
    std::vector<std::string> names;
    std::vector<int64_t> chrom_len;
    std::vector<int64_t> chrom_ptr;     // n_chrom + 1: items of chromosome c are [ptr[c], ptr[c+1])
    int64_t n_items = 0;
    int32_t* start = nullptr;           // 1-based closed
    int32_t* end = nullptr;
    uint32_t* value = nullptr;          // float bits, -0.0 stored as +0.0
    int64_t* d_chrom_ptr = nullptr;
    int64_t* d_chrom_len = nullptr;
};

std::map<int, std::unique_ptr<Signal>> g_signals;
int g_next_signal = 1;

void signal_release(Signal& s) {
    dfree(s.start);
    dfree(s.end);
    dfree(s.value);
    dfree(s.d_chrom_ptr);
    dfree(s.d_chrom_len);
}

Signal* get_signal(int h) {
    auto it = g_signals.find(h);
    return it == g_signals.end() ? nullptr : it->second.get();
}

// ---- host parse ------------------------------------------------------------------------------
struct Reader {
    const uint8_t* d;
    int64_t n;
    bool ok(int64_t off, int64_t bytes) const { return off >= 0 && bytes >= 0 && off <= n && bytes <= n - off; }
    uint32_t u8(int64_t o) const { return d[o]; }
    uint32_t u16(int64_t o) const { return (uint32_t)d[o] | ((uint32_t)d[o + 1] << 8); }
    uint32_t u32(int64_t o) const { return u16(o) | (u16(o + 2) << 16); }
    uint64_t u64(int64_t o) const { return (uint64_t)u32(o) | ((uint64_t)u32(o + 4) << 32); }
};

int truncated(const char* what, int64_t off) {
    return fail(RCP_ERR_DATA, "bigWig: truncated file (%s at byte %lld runs past the end)", what, (long long)off);
}

// chromosome B+ tree (bbiFile.h bptFile): leaves hold (key, chromId, chromSize)
int walk_chrom_tree(const Reader& r, int64_t node, uint32_t key_size, int depth, std::vector<std::string>* names,
                    std::vector<int64_t>* sizes, std::vector<uint8_t>* seen) {
    if (depth > 64) return fail(RCP_ERR_DATA, "bigWig: the chromosome tree is deeper than 64 levels");
    if (!r.ok(node, 4)) return truncated("chromosome tree node", node);
    const bool leaf = r.u8(node) != 0;
    const uint32_t count = r.u16(node + 2);
    const int64_t item = (int64_t)key_size + 8;
    if (!r.ok(node + 4, item * count)) return truncated("chromosome tree node", node);
    for (uint32_t i = 0; i < count; i++) {
        const int64_t p = node + 4 + item * i;
        if (leaf) {
            size_t len = 0;
            while (len < key_size && r.d[p + len] != 0) len++;     // keys are NUL-padded to keySize
            const uint32_t id = r.u32(p + key_size), size = r.u32(p + key_size + 4);
            if (id >= names->size() || (*seen)[id])
                return fail(RCP_ERR_DATA, "bigWig: chromosome id %u is out of range or repeated", id);
            if (size > 0x7fffffffu)
                return fail(RCP_ERR_UNSUPPORTED, "bigWig: chromosome size %u exceeds 32-bit coordinates", size);
            (*seen)[id] = 1;
            (*names)[id].assign(reinterpret_cast<const char*>(r.d + p), len);
            (*sizes)[id] = size;
        } else {
            RCP_TRY(walk_chrom_tree(r, (int64_t)r.u64(p + key_size), key_size, depth + 1, names, sizes, seen));
        }
    }
    return RCP_OK;
}

// R-tree index (cirTree.h): leaves hold (startChrom, startBase, endChrom, endBase, offset, size)
int walk_rtree(const Reader& r, int64_t node, int depth, std::vector<InflateJob>* blocks) {
    if (depth > 64) return fail(RCP_ERR_DATA, "bigWig: the R-tree is deeper than 64 levels");
    if (!r.ok(node, 4)) return truncated("R-tree node", node);
    const bool leaf = r.u8(node) != 0;
    const uint32_t count = r.u16(node + 2);
    const int64_t item = leaf ? 32 : 24;
    if (!r.ok(node + 4, item * count)) return truncated("R-tree node", node);
    for (uint32_t i = 0; i < count; i++) {
        const int64_t p = node + 4 + item * i;
        if (leaf) {
            InflateJob b;
            b.in_off = (int64_t)r.u64(p + 16);
            b.in_len = (int64_t)r.u64(p + 24);
            if (!r.ok(b.in_off, b.in_len)) return truncated("data block", b.in_off);
            blocks->push_back(b);
        } else {
            RCP_TRY(walk_rtree(r, (int64_t)r.u64(p + 16), depth + 1, blocks));
        }
    }
    return RCP_OK;
}

// ---- device expand + validation ------------------------------------------------------------------
// error key: (block << 20) | (item << 4) | code, the smallest wins (first block, first item)
enum {
    E_SHORT = 1,       // section shorter than its 24-byte header
    E_SIZE = 2,        // section size != header + itemCount * item size
    E_TYPE = 3,        // unknown section type
    E_CHROM = 4,       // chromId not in the chromosome tree
    E_EMPTY = 5,       // item end <= start (0-based half-open)
    E_PAST = 6,        // item end past chromSize
    E_VALUE = 7,       // NaN or infinite value
    E_ORDER = 8,       // items not sorted / overlapping within a chromosome
    E_BLOCK = 9        // a block inflates past uncompressBufSize (set on the host)
};

__device__ __forceinline__ void report(unsigned long long* err, int64_t block, uint32_t item, unsigned code) {
    atomicMin(err, ((unsigned long long)block << 20) | ((unsigned long long)item << 4) | code);
}

// One CTA per data block (one section each).
__global__ void __launch_bounds__(256)
bw_expand_kernel(const uint8_t* __restrict__ buf, const int64_t* __restrict__ boff, const uint32_t* __restrict__ blen,
                 const int64_t* __restrict__ item_off, int n_chrom, const int64_t* __restrict__ chrom_len,
                 int32_t* __restrict__ it_start, int32_t* __restrict__ it_end, uint32_t* __restrict__ it_val,
                 unsigned long long* __restrict__ err) {
    const int64_t b = blockIdx.x;
    const uint8_t* s = buf + boff[b];
    const uint32_t len = blen[b];
    const int64_t o = item_off[b];
    const uint32_t n_host = (uint32_t)(item_off[b + 1] - o);
    auto rd32 = [&](uint32_t at) {
        return (uint32_t)s[at] | ((uint32_t)s[at + 1] << 8) | ((uint32_t)s[at + 2] << 16) | ((uint32_t)s[at + 3] << 24);
    };
    if (len < SECTION_HEAD) {
        if (threadIdx.x == 0) report(err, b, 0, E_SHORT);
        return;
    }
    const uint32_t chrom = rd32(0), sec_start = rd32(4), step = rd32(12), span = rd32(16);
    const uint32_t type = s[20];
    const uint32_t count = (uint32_t)s[22] | ((uint32_t)s[23] << 8);
    const uint32_t isz = type == 1 ? 12u : type == 2 ? 8u : type == 3 ? 4u : 0u;
    if (threadIdx.x == 0) {
        if (isz == 0) report(err, b, 0, E_TYPE);
        else if (len != SECTION_HEAD + isz * count || count != n_host) report(err, b, 0, E_SIZE);
        else if (chrom >= (uint32_t)n_chrom) report(err, b, 0, E_CHROM);
    }
    if (isz == 0 || len != SECTION_HEAD + isz * count || count != n_host || chrom >= (uint32_t)n_chrom) return;
    const int64_t clen = chrom_len[chrom];
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) {
        const uint8_t* it = s + SECTION_HEAD + (size_t)i * isz;
        uint32_t s0, e0, vb;
        auto r32 = [&](int at) {
            return (uint32_t)it[at] | ((uint32_t)it[at + 1] << 8) | ((uint32_t)it[at + 2] << 16) |
                   ((uint32_t)it[at + 3] << 24);
        };
        if (type == 1) {            // bedGraph: start, end, value
            s0 = r32(0);
            e0 = r32(4);
            vb = r32(8);
        } else if (type == 2) {     // varStep: start, value; span = itemSpan
            s0 = r32(0);
            e0 = s0 + span;
            vb = r32(4);
        } else {                    // fixedStep: value; start = secStart + i * itemStep
            s0 = sec_start + i * step;
            e0 = s0 + span;
            vb = r32(0);
        }
        float v = __uint_as_float(vb);
        if (!isfinite(v)) report(err, b, i, E_VALUE);
        if (v == 0.0f) vb = 0u;     // -0.0 -> +0.0: equal bits <=> equal values
        if (type != 1 && (uint64_t)s0 + span > 0xffffffffull) report(err, b, i, E_PAST);
        else if (e0 <= s0) report(err, b, i, E_EMPTY);
        else if ((int64_t)e0 > clen) report(err, b, i, E_PAST);
        it_start[o + i] = (int32_t)(s0 + 1u);
        it_end[o + i] = (int32_t)e0;
        it_val[o + i] = vb;
    }
    __syncthreads();                // the CTA's own stores are visible to it
    for (uint32_t i = threadIdx.x + 1; i < count; i += blockDim.x)
        if (it_start[o + i] <= it_end[o + i - 1]) report(err, b, i, E_ORDER);
}

// Order across blocks: chromosome ids never decrease, and the first item of a block starts after
// the last item of the previous non-empty block on the same chromosome.
__global__ void __launch_bounds__(256)
bw_order_kernel(int64_t nb, const uint8_t* __restrict__ buf, const int64_t* __restrict__ boff,
                const uint32_t* __restrict__ blen, const int64_t* __restrict__ item_off,
                const int32_t* __restrict__ it_start, const int32_t* __restrict__ it_end,
                unsigned long long* __restrict__ err) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b <= 0 || b >= nb) return;
    const int64_t k = item_off[b];
    if (item_off[b + 1] == k || k == 0) return;                 // empty block, or nothing before it
    int64_t lo = 0, hi = b;                                     // last block p < b with items
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (item_off[mid] <= k - 1) lo = mid;
        else hi = mid - 1;
    }
    const int64_t p = lo;
    if (blen[b] < SECTION_HEAD || blen[p] < SECTION_HEAD) return;   // reported by the expand kernel
    auto chrom_of = [&](int64_t q) {
        const uint8_t* s = buf + boff[q];
        return (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
    };
    const uint32_t cb = chrom_of(b), cp = chrom_of(p);
    if (cb < cp || (cb == cp && it_start[k] <= it_end[k - 1])) report(err, b, 0, E_ORDER);
}

// ---- coverage ------------------------------------------------------------------------------------
constexpr int SCTA = 256;
constexpr int SWARPS = SCTA / 32;
constexpr int ST = 1024;            // positions per warp tile (4 KB of shared memory)

// One thread per element: the R subscript rules of `cov[i2k]` (coverage.R:202-209 inside the
// tryCatch of 217-222), the element's length, and the pieces (one per range) with their tiles.
__global__ void __launch_bounds__(SCTA)
sig_plan_kernel(int64_t G, const int64_t* __restrict__ ptr, const int32_t* __restrict__ chrom,
                const int32_t* __restrict__ start, const int32_t* __restrict__ end, int n_chrom,
                const int64_t* __restrict__ chrom_len, int32_t* __restrict__ len, uint8_t* __restrict__ is_null,
                int64_t* __restrict__ padded, int64_t* __restrict__ p_elem, int32_t* __restrict__ p_gs,
                int32_t* __restrict__ p_w, int32_t* __restrict__ p_prefix, int64_t* __restrict__ p_tiles,
                unsigned int* __restrict__ err, unsigned long long* __restrict__ stats) {
    const int64_t g = (int64_t)blockIdx.x * SCTA + threadIdx.x;
    unsigned long long my_null = 0, my_len = 0;
    if (g < G) {
        const int64_t a = ptr ? ptr[g] : g, b = ptr ? ptr[g + 1] : g + 1;
        bool null = b <= a;
        const int c = null ? -1 : chrom[a];
        if (!null && (c < -1 || c >= n_chrom)) {
            atomicOr(err, 1u);
            null = true;
        }
        if (c < 0) null = true;                                 // not in the track
        const int64_t clen = c >= 0 ? chrom_len[c] : 0;
        for (int64_t j = a; j < b; j++) {
            const int64_t s = start[j], e = end[j];
            if (e < s - 1) {
                atomicOr(err, 2u);
                null = true;
            } else if (e >= s && (s < 0 || e > clen)) {
                null = true;                                    // negative or out-of-bounds subscript
            }
        }
        int64_t L = 0;
        for (int64_t j = a; j < b; j++) {
            const int64_t s = start[j] > 1 ? start[j] : 1, e = end[j];   // a 0 subscript is dropped
            const int64_t w = null ? 0 : (e >= s ? e - s + 1 : 0);
            p_elem[j] = g;
            p_gs[j] = (int32_t)s;
            p_w[j] = (int32_t)w;
            p_prefix[j] = (int32_t)L;
            p_tiles[j] = (w + ST - 1) / ST;
            L += w;
        }
        if (L > 0x7fffffffll) {
            atomicOr(err, 4u);
            L = 0;
        }
        if (L == 0) {
            null = true;
            for (int64_t j = a; j < b; j++) p_tiles[j] = 0;
        }
        len[g] = null ? 0 : (int32_t)L;
        is_null[g] = null ? 1 : 0;
        padded[g] = null ? 0 : ((L + covk::PAD - 1) / covk::PAD) * covk::PAD;
        my_null = null ? 1 : 0;
        my_len = null ? 0 : (unsigned long long)L;
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

struct SigTileArgs {
    int64_t n_tiles, n_ranges;
    const int64_t* tile_off;        // n_ranges + 1
    const int64_t* p_elem;
    const int32_t* p_gs;
    const int32_t* p_w;
    const int32_t* p_prefix;
    const int64_t* ptr;             // nullptr: range g is element g
    const int32_t* chrom;
    const int8_t* strand;           // nullptr: all '*'
    const int64_t* off;
    const int32_t* len;
    const int64_t* chrom_ptr;
    const int32_t* it_start;
    const int32_t* it_end;
    const uint32_t* it_val;
    uint32_t* cov;
};

__global__ void __launch_bounds__(SCTA) sig_tile_kernel(SigTileArgs p) {
    __shared__ uint32_t tiles[SWARPS][ST];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* tile = tiles[warp];
    const int64_t n_warps = (int64_t)gridDim.x * SWARPS;
    for (int64_t t = (int64_t)blockIdx.x * SWARPS + warp; t < p.n_tiles; t += n_warps) {
        int64_t lo = 0, hi = p.n_ranges - 1;                    // the range j that owns tile t
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (__ldg(p.tile_off + mid + 1) <= t) lo = mid + 1;
            else hi = mid;
        }
        const int64_t j = lo;
        const int64_t g = __ldg(p.p_elem + j);
        const int64_t a = p.ptr ? __ldg(p.ptr + g) : g;
        const int c = __ldg(p.chrom + a);
        const bool rev = p.strand && __ldg(p.strand + a) < 0;
        const int k0 = (int)(t - __ldg(p.tile_off + j)) * ST;
        const int n = min(ST, __ldg(p.p_w + j) - k0);
        const int gp0 = __ldg(p.p_gs + j) + k0, gp1 = gp0 + n - 1;
        for (int q = lane; q < n; q += 32) tile[q] = 0u;
        // first item that ends at or after gp0
        int64_t i = __ldg(p.chrom_ptr + c), i1 = __ldg(p.chrom_ptr + c + 1);
        {
            int64_t b = i1;
            while (i < b) {
                const int64_t mid = (i + b) >> 1;
                if (__ldg(p.it_end + mid) < gp0) i = mid + 1;
                else b = mid;
            }
        }
        __syncwarp();
        while (i < i1) {
            const int64_t k = i + lane;
            int s = 0x7fffffff, e = 0;
            uint32_t v = 0;
            if (k < i1) {
                s = __ldg(p.it_start + k);
                e = __ldg(p.it_end + k);
                v = __ldg(p.it_val + k);
            }
            const unsigned in = __ballot_sync(0xffffffffu, s <= gp1);    // sorted: a prefix of the lanes
            const int cnt = __popc(in);
            for (int u = 0; u < cnt; u++) {
                const int su = __shfl_sync(0xffffffffu, s, u), eu = __shfl_sync(0xffffffffu, e, u);
                const uint32_t vu = __shfl_sync(0xffffffffu, v, u);
                const int qa = max(su, gp0) - gp0, qb = min(eu, gp1) - gp0;
                for (int q = qa + lane; q <= qb; q += 32) tile[q] = vu;
            }
            if (cnt < 32) break;
            i += 32;
        }
        __syncwarp();
        const int64_t base = __ldg(p.off + g);
        const int64_t L = __ldg(p.len + g);
        const int64_t kf0 = (int64_t)__ldg(p.p_prefix + j) + k0;
        uint32_t* dst = p.cov + base;
        if (!rev) {
            for (int q = lane; q < n; q += 32) dst[kf0 + q] = tile[q];
        } else {
            for (int q = lane; q < n; q += 32) dst[L - 1 - (kf0 + q)] = tile[q];
        }
        __syncwarp();
    }
}

}  // namespace

void signal_release_all() {
    for (auto& kv : g_signals) signal_release(*kv.second);
    g_signals.clear();
}

}  // namespace rcp

using namespace rcp;

extern "C" {

int rcp_bigwig_load(const uint8_t* data, int64_t n_bytes, int n_threads, int* signal_out) {
    RCP_TRY(require_ready());
    if (n_bytes < 0 || (n_bytes > 0 && data == nullptr) || signal_out == nullptr)
        return fail(RCP_ERR_ARG, "rcp_bigwig_load: bad argument");
    const Reader r{data, n_bytes};
    if (!r.ok(0, 4)) return truncated("header", 0);
    const uint32_t magic = r.u32(0);
    if (magic == BIGBED_MAGIC) return fail(RCP_ERR_DATA, "bigWig: the file is bigBed, not bigWig");
    if (magic == __builtin_bswap32(BIGWIG_MAGIC))
        return fail(RCP_ERR_UNSUPPORTED, "bigWig: big-endian files are not supported");
    if (magic != BIGWIG_MAGIC) return fail(RCP_ERR_DATA, "bigWig: bad magic 0x%08x (not a bigWig file)", magic);
    if (!r.ok(0, 64)) return truncated("header", 0);
    const uint32_t zoom_levels = r.u16(6);
    const int64_t chrom_tree = (int64_t)r.u64(8), index = (int64_t)r.u64(24);
    const uint32_t buf_size = r.u32(52);
    if (!r.ok(64, 24ll * zoom_levels)) return truncated("zoom headers", 64);   // skipped
    // chromosome B+ tree
    if (!r.ok(chrom_tree, 32)) return truncated("chromosome tree header", chrom_tree);
    if (r.u32(chrom_tree) != CHROM_TREE_MAGIC)
        return fail(RCP_ERR_DATA, "bigWig: bad chromosome tree magic 0x%08x", r.u32(chrom_tree));
    const uint32_t key_size = r.u32(chrom_tree + 8), val_size = r.u32(chrom_tree + 12);
    const uint64_t n_chrom64 = r.u64(chrom_tree + 16);
    if (val_size != 8 || key_size == 0 || key_size > 255 || n_chrom64 > (uint64_t)(n_bytes / 8 + 1))
        return fail(RCP_ERR_DATA, "bigWig: bad chromosome tree header (keySize %u, valSize %u, %llu chromosomes)",
                    key_size, val_size, (unsigned long long)n_chrom64);
    const int n_chrom = (int)n_chrom64;
    std::unique_ptr<Signal> sig(new Signal());
    sig->n_chrom = n_chrom;
    sig->names.resize((size_t)n_chrom);
    sig->chrom_len.assign((size_t)n_chrom, 0);
    std::vector<uint8_t> seen((size_t)n_chrom, 0);
    RCP_TRY(walk_chrom_tree(r, chrom_tree + 32, key_size, 0, &sig->names, &sig->chrom_len, &seen));
    for (int c = 0; c < n_chrom; c++)
        if (!seen[(size_t)c]) return fail(RCP_ERR_DATA, "bigWig: the chromosome tree has no chromosome id %d", c);
    // R-tree index -> data blocks in file order
    if (!r.ok(index, 48)) return truncated("R-tree header", index);
    if (r.u32(index) != RTREE_MAGIC) return fail(RCP_ERR_DATA, "bigWig: bad R-tree magic 0x%08x", r.u32(index));
    std::vector<InflateJob> jobs;
    RCP_TRY(walk_rtree(r, index + 48, 0, &jobs));
    const int64_t nb = (int64_t)jobs.size();
    int64_t cap_total = 0;
    for (auto& j : jobs) {
        if (buf_size == 0 && j.in_len > 0xffffffffll)
            return fail(RCP_ERR_DATA, "bigWig: a data block of %lld bytes", (long long)j.in_len);
        j.out_off = cap_total;
        j.out_cap = buf_size > 0 ? buf_size : (uint32_t)j.in_len;
        cap_total += j.out_cap;
    }
    std::unique_ptr<uint8_t[]> host(new uint8_t[(size_t)std::max<int64_t>(cap_total, 1)]);
    const int64_t bad = inflate_jobs(data, jobs.data(), nb, host.get(), n_threads, buf_size > 0 ? INFLATE_ZLIB : INFLATE_COPY);
    if (bad == -2) return fail(RCP_ERR_CUDA, "rcp_bigwig_load: zlib could not be initialised");
    if (bad >= 0)
        return fail(RCP_ERR_DATA, "bigWig: data block %lld (file byte %lld) does not inflate to at most %u bytes",
                    (long long)bad, (long long)jobs[(size_t)bad].in_off, buf_size);
    // item counts (sizes the arrays; the device checks them against the section sizes) and the
    // per-chromosome item ranges (valid once the device has checked the order)
    std::vector<int64_t> boff((size_t)nb), item_off((size_t)nb + 1, 0);
    std::vector<uint32_t> blen((size_t)nb);
    std::vector<int64_t> per_chrom((size_t)n_chrom + 1, 0);
    for (int64_t b = 0; b < nb; b++) {
        const InflateJob& j = jobs[(size_t)b];
        boff[(size_t)b] = j.out_off;
        blen[(size_t)b] = j.out_len;
        const uint8_t* s = host.get() + j.out_off;
        int64_t cnt = 0;
        if (j.out_len >= (uint32_t)SECTION_HEAD) {
            cnt = (int64_t)s[22] | ((int64_t)s[23] << 8);
            const uint32_t c = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
            if (c < (uint32_t)n_chrom) per_chrom[c] += cnt;
        }
        item_off[(size_t)b + 1] = item_off[(size_t)b] + cnt;
    }
    sig->n_items = item_off[(size_t)nb];
    if (sig->n_items > 0x7fffffffll * 8)
        return fail(RCP_ERR_UNSUPPORTED, "bigWig: %lld items", (long long)sig->n_items);
    sig->chrom_ptr.assign((size_t)n_chrom + 1, 0);
    for (int c = 0; c < n_chrom; c++) sig->chrom_ptr[(size_t)c + 1] = sig->chrom_ptr[(size_t)c] + per_chrom[(size_t)c];
    // device: upload once, expand, validate
    uint8_t* d_buf = nullptr;
    int64_t *d_boff = nullptr, *d_item_off = nullptr;
    uint32_t* d_blen = nullptr;
    unsigned long long* d_err = nullptr;
    auto cleanup = [&]() {
        dfree(d_buf);
        dfree(d_boff);
        dfree(d_item_off);
        dfree(d_blen);
        dfree(d_err);
    };
    int rc = RCP_OK;
    auto step = [&](int e) {
        if (rc == RCP_OK) rc = e;
    };
    step(dalloc(&d_buf, (size_t)cap_total));
    step(dalloc(&d_boff, (size_t)nb));
    step(dalloc(&d_item_off, (size_t)nb + 1));
    step(dalloc(&d_blen, (size_t)nb));
    step(dalloc(&d_err, 1));
    step(dalloc(&sig->start, (size_t)sig->n_items));
    step(dalloc(&sig->end, (size_t)sig->n_items));
    step(dalloc(&sig->value, (size_t)sig->n_items));
    step(dalloc(&sig->d_chrom_ptr, (size_t)n_chrom + 1));
    step(dalloc(&sig->d_chrom_len, (size_t)n_chrom));
    auto h2d = [&](void* dst, const void* src, size_t bytes) {
        if (rc == RCP_OK && bytes > 0) {
            const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream);
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "bigWig upload failed: %s", cudaGetErrorString(e));
        }
    };
    h2d(d_buf, host.get(), (size_t)cap_total);
    h2d(d_boff, boff.data(), (size_t)nb * 8);
    h2d(d_item_off, item_off.data(), ((size_t)nb + 1) * 8);
    h2d(d_blen, blen.data(), (size_t)nb * 4);
    h2d(sig->d_chrom_ptr, sig->chrom_ptr.data(), ((size_t)n_chrom + 1) * 8);
    h2d(sig->d_chrom_len, sig->chrom_len.data(), (size_t)n_chrom * 8);
    if (rc == RCP_OK && cudaMemsetAsync(d_err, 0xff, 8, g_ctx.stream) != cudaSuccess)
        rc = fail(RCP_ERR_CUDA, "bigWig: memset failed");
    unsigned long long h_err = ~0ull;
    if (rc == RCP_OK && nb > 0) {
        bw_expand_kernel<<<(unsigned)nb, 256, 0, g_ctx.stream>>>(d_buf, d_boff, d_blen, d_item_off, n_chrom,
                                                                 sig->d_chrom_len, sig->start, sig->end, sig->value,
                                                                 d_err);
        g_ctx.launches++;
        bw_order_kernel<<<blocks_for(nb, 256), 256, 0, g_ctx.stream>>>(nb, d_buf, d_boff, d_blen, d_item_off,
                                                                        sig->start, sig->end, d_err);
        g_ctx.launches++;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "bigWig expand launch failed: %s", cudaGetErrorString(e));
    }
    if (rc == RCP_OK) {
        const FetchItem items[1] = {{d_err, &h_err, 8}};
        rc = fetch_and_sync(items, 1);
    }
    if (rc == RCP_OK && h_err != ~0ull) {
        static const char* const what[] = {"",
                                           "the section is shorter than its 24-byte header",
                                           "the section size disagrees with its item count",
                                           "unknown section type (not bedGraph, varStep or fixedStep)",
                                           "the section's chromId is not in the chromosome tree",
                                           "end <= start",
                                           "the item ends past chromSize",
                                           "the value is NaN or infinite",
                                           "the items of a chromosome are not sorted and disjoint"};
        const int64_t b = (int64_t)(h_err >> 20);
        const unsigned item = (unsigned)((h_err >> 4) & 0xffffu), code = (unsigned)(h_err & 15u);
        const uint8_t* s = host.get() + jobs[(size_t)b].out_off;
        std::string chrom = "?";
        if (jobs[(size_t)b].out_len >= 4) {
            const uint32_t c = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
            if (c < (uint32_t)n_chrom) chrom = sig->names[c];
        }
        rc = fail(RCP_ERR_DATA, "bigWig: data block %lld (chromosome %s), item %u: %s", (long long)b, chrom.c_str(),
                  item, code < 9 ? what[code] : "bad data");
    }
    cleanup();
    if (rc != RCP_OK) {
        signal_release(*sig);
        return rc;
    }
    const int h = g_next_signal++;
    g_signals[h] = std::move(sig);
    *signal_out = h;
    return RCP_OK;
}

int rcp_signal_info(int signal, int* n_chrom, int64_t* n_items, int64_t* names_bytes) {
    Signal* s = get_signal(signal);
    if (!s) return fail(RCP_ERR_HANDLE, "unknown signal handle %d", signal);
    if (n_chrom) *n_chrom = s->n_chrom;
    if (n_items) *n_items = s->n_items;
    if (names_bytes) {
        int64_t t = 0;
        for (auto& nm : s->names) t += (int64_t)nm.size() + 1;
        *names_bytes = t;
    }
    return RCP_OK;
}

int rcp_signal_chroms(int signal, char* names, int64_t* chrom_len) {
    Signal* s = get_signal(signal);
    if (!s) return fail(RCP_ERR_HANDLE, "unknown signal handle %d", signal);
    if (names) {
        for (auto& nm : s->names) {
            memcpy(names, nm.c_str(), nm.size() + 1);
            names += nm.size() + 1;
        }
    }
    if (chrom_len) memcpy(chrom_len, s->chrom_len.data(), s->chrom_len.size() * 8);
    return RCP_OK;
}

int rcp_signal_fetch(int signal, int32_t* chrom, int32_t* start, int32_t* end, float* value, int64_t capacity) {
    RCP_TRY(require_ready());
    Signal* s = get_signal(signal);
    if (!s) return fail(RCP_ERR_HANDLE, "unknown signal handle %d", signal);
    if (capacity < s->n_items) return fail(RCP_ERR_ARG, "rcp_signal_fetch: %lld items, capacity %lld",
                                           (long long)s->n_items, (long long)capacity);
    const size_t n = (size_t)s->n_items;
    if (n == 0) return RCP_OK;
    if (start) RCP_CUDA(cudaMemcpyAsync(start, s->start, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (end) RCP_CUDA(cudaMemcpyAsync(end, s->end, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (value) RCP_CUDA(cudaMemcpyAsync(value, s->value, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    if (chrom)
        for (int c = 0; c < s->n_chrom; c++)
            for (int64_t k = s->chrom_ptr[(size_t)c]; k < s->chrom_ptr[(size_t)c + 1]; k++) chrom[k] = c;
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return RCP_OK;
}

int rcp_signal_free(int signal) {
    auto it = g_signals.find(signal);
    if (it == g_signals.end()) return fail(RCP_ERR_HANDLE, "unknown signal handle %d", signal);
    signal_release(*it->second);
    g_signals.erase(it);
    return RCP_OK;
}

int rcp_signal_coverage(int signal, int64_t n_elements, const int64_t* ptr, const int32_t* chrom, const int32_t* start,
                        const int32_t* end, const int8_t* strand, int mem, int* cov_out) {
    RCP_TRY(require_ready());
    Signal* sg = get_signal(signal);
    if (!sg) return fail(RCP_ERR_HANDLE, "unknown signal handle %d", signal);
    if (n_elements < 0 || cov_out == nullptr || (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE))
        return fail(RCP_ERR_ARG, "rcp_signal_coverage: bad argument");
    int64_t n_ranges = n_elements;
    if (ptr) {
        if (mem != RCP_MEM_HOST)
            return fail(RCP_ERR_UNSUPPORTED, "rcp_signal_coverage takes a host ptr (it is read on the host)");
        if (ptr[0] != 0) return fail(RCP_ERR_ARG, "ptr[0] must be 0");
        for (int64_t g = 0; g < n_elements; g++)
            if (ptr[g + 1] < ptr[g]) return fail(RCP_ERR_ARG, "ptr is not non-decreasing at %lld", (long long)g);
        n_ranges = ptr[n_elements];
    }
    if (n_ranges > 0 && (!chrom || !start || !end)) return fail(RCP_ERR_ARG, "rcp_signal_coverage: NULL array");
    const int64_t G = n_elements;
    DevIn<int64_t> d_ptr;
    DevIn<int32_t> d_chrom, d_start, d_end;
    DevIn<int8_t> d_strand;
    RCP_TRY(d_ptr.init(ptr, (size_t)G + 1, ptr ? RCP_MEM_HOST : mem));
    RCP_TRY(d_chrom.init(chrom, (size_t)n_ranges, mem));
    RCP_TRY(d_start.init(start, (size_t)n_ranges, mem));
    RCP_TRY(d_end.init(end, (size_t)n_ranges, mem));
    RCP_TRY(d_strand.init(strand, (size_t)n_ranges, mem));
    Coverage* cv;
    int h;
    RCP_TRY(new_coverage(&cv, &h));
    cv->value_type = RCP_VALUE_FLOAT32;
    cv->n_regions = G;
    int64_t *padded = nullptr, *p_elem = nullptr, *p_tiles = nullptr, *tile_off = nullptr;
    int32_t *p_gs = nullptr, *p_w = nullptr, *p_prefix = nullptr;
    unsigned int* d_err = nullptr;
    unsigned long long* d_stats = nullptr;
    int rc = RCP_OK;
    auto step = [&](int e) {
        if (rc == RCP_OK) rc = e;
    };
    step(dalloc(&cv->off, (size_t)G + 1));
    step(dalloc(&cv->len, (size_t)G));
    step(dalloc(&cv->is_null, (size_t)G));
    step(dalloc(&padded, (size_t)G));
    step(dalloc(&p_elem, (size_t)n_ranges));
    step(dalloc(&p_gs, (size_t)n_ranges));
    step(dalloc(&p_w, (size_t)n_ranges));
    step(dalloc(&p_prefix, (size_t)n_ranges));
    step(dalloc(&p_tiles, (size_t)n_ranges));
    step(dalloc(&tile_off, (size_t)n_ranges + 1));
    step(dalloc(&d_err, 1));
    step(dalloc(&d_stats, 3));
    if (rc == RCP_OK && (cudaMemsetAsync(d_err, 0, 4, g_ctx.stream) != cudaSuccess ||
                         cudaMemsetAsync(d_stats, 0, 24, g_ctx.stream) != cudaSuccess))
        rc = fail(RCP_ERR_CUDA, "rcp_signal_coverage: memset failed");
    struct {
        int64_t total_padded, n_tiles;
        unsigned long long stats[3];
        unsigned int err;
    } hs = {0, 0, {0, 0, 0}, 0};
    if (rc == RCP_OK) {
        StageTimer plan_timer(ST_COV_LIST);
        if (G > 0) {
            sig_plan_kernel<<<blocks_for(G, SCTA), SCTA, 0, g_ctx.stream>>>(
                G, d_ptr.ptr, d_chrom.ptr, d_start.ptr, d_end.ptr, sg->n_chrom, sg->d_chrom_len, cv->len, cv->is_null,
                padded, p_elem, p_gs, p_w, p_prefix, p_tiles, d_err, d_stats);
            g_ctx.launches++;
            if (cudaGetLastError() != cudaSuccess) rc = fail(RCP_ERR_CUDA, "signal plan kernel launch failed");
        }
        if (G == n_ranges) {
            step(exclusive_scan2_i64(padded, cv->off, cv->off + G, p_tiles, tile_off, tile_off + G, G));
        } else {
            step(exclusive_scan_i64(padded, cv->off, G, cv->off + G));
            step(exclusive_scan_i64(p_tiles, tile_off, n_ranges, tile_off + n_ranges));
        }
    }
    if (rc == RCP_OK) {
        const FetchItem items[4] = {{cv->off + G, &hs.total_padded, 8}, {tile_off + n_ranges, &hs.n_tiles, 8},
                                    {d_stats, hs.stats, 24}, {d_err, &hs.err, 4}};
        rc = fetch_and_sync(items, 4);
    }
    if (rc == RCP_OK) {
        if (hs.err & 1u) rc = fail(RCP_ERR_DATA, "a range has a chromosome id outside [-1, n_chrom)");
        else if (hs.err & 2u) rc = fail(RCP_ERR_DATA, "a range has end < start - 1");
        else if (hs.err & 4u) rc = fail(RCP_ERR_UNSUPPORTED, "an element is longer than 2^31 - 1 positions");
    }
    if (rc == RCP_OK) {
        cv->total_padded = hs.total_padded;
        cv->n_null = (int64_t)hs.stats[0];
        cv->total_len = (int64_t)hs.stats[1];
        cv->max_len = (int32_t)hs.stats[2];
        rc = dalloc(&cv->cov, (size_t)hs.total_padded);
    }
    if (rc == RCP_OK && hs.n_tiles > 0) {
        StageTimer tile_timer(ST_COV_TILE);
        SigTileArgs a;
        a.n_tiles = hs.n_tiles;
        a.n_ranges = n_ranges;
        a.tile_off = tile_off;
        a.p_elem = p_elem;
        a.p_gs = p_gs;
        a.p_w = p_w;
        a.p_prefix = p_prefix;
        a.ptr = d_ptr.ptr;
        a.chrom = d_chrom.ptr;
        a.strand = d_strand.ptr;
        a.off = cv->off;
        a.len = cv->len;
        a.chrom_ptr = sg->d_chrom_ptr;
        a.it_start = sg->start;
        a.it_end = sg->end;
        a.it_val = sg->value;
        a.cov = reinterpret_cast<uint32_t*>(cv->cov);
        const int64_t ctas = std::min<int64_t>((hs.n_tiles + SWARPS - 1) / SWARPS, (int64_t)g_ctx.sm_count * 8);
        sig_tile_kernel<<<(unsigned)ctas, SCTA, 0, g_ctx.stream>>>(a);
        g_ctx.launches++;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "signal tile kernel launch failed: %s", cudaGetErrorString(e));
    }
    dfree(padded);
    dfree(p_elem);
    dfree(p_gs);
    dfree(p_w);
    dfree(p_prefix);
    dfree(p_tiles);
    dfree(tile_off);
    dfree(d_err);
    dfree(d_stats);
    if (rc != RCP_OK) {
        rcp_coverage_free(h);
        return rc;
    }
    *cov_out = h;
    return RCP_OK;
}

}  // extern "C"
