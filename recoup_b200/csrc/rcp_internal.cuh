// Internal declarations shared by the translation units of librecoup_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "recoup_b200.h"

namespace rcp {

// ------------------------------------------------------------------ context / errors -------
struct Ctx {
    bool ready = false;
    int device = -1;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t mem_bytes = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;      // kernels launched by this library
    int coverage_path = RCP_PATH_AUTO;
    bool deferred_validation = false;   // rcp_set_deferred_validation
};
extern Ctx g_ctx;

int fail(int code, const char* fmt, ...);   // records the message, returns code
constexpr int RCP_SWITCH_TO_INDEX = -1000;   // internal: the bucket path hands the call to the index path
constexpr int RCP_SPLIT_NOT_APPLICABLE = -1001;   // internal: the split path cannot serve this call
int require_ready();                         // RCP_OK or RCP_ERR_NOGPU

#define RCP_CUDA(call)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess)                                                                 \
            return ::rcp::fail(RCP_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__,        \
                               __LINE__, cudaGetErrorString(_e));                              \
    } while (0)

#define RCP_TRY(expr)                                                                          \
    do {                                                                                       \
        int _rc = (expr);                                                                      \
        if (_rc != RCP_OK) return _rc;                                                         \
    } while (0)

#define RCP_LAUNCHED()                                                                         \
    do {                                                                                       \
        ::rcp::g_ctx.launches++;                                                               \
        RCP_CUDA(cudaGetLastError());                                                          \
    } while (0)

// ------------------------------------------------------------------ stage timers -----------
// Optional CUDA-event timing of the library's own stages on the library stream (used by
// bench.py for the roofline object).  Off by default; when off a StageTimer does nothing.
enum Stage {
    ST_INDEX_MAP = 0,   // reads -> global coordinates (+ strand compaction)
    ST_INDEX_SORT,      // radix sorts of the index
    ST_COV_PLAN,        // region plan kernel + offset scans + tile list
    ST_COV_TILE,        // cov_tile_kernel
    ST_COV_SMALL,       // cov_small_kernel
    ST_COV_LIST,        // list plan + cov_list_kernel
    ST_COV_CONCAT,      // c(left, center, right)
    ST_PROF_BIN,        // bin_matrix_kernel
    ST_PROF_INTERP,     // interp_kernel
    ST_PROF_BASE,       // base_matrix_kernel
    ST_FUSED,           // fused coverage+profile kernel
    ST_BKT_PLAN,        // bucket path: windows, tiles, cell lists, NULL rule, offset scans
    ST_BKT_COUNT,       // bucket path: count pass over the reads
    ST_BKT_SCATTER,     // bucket path: scatter pass over the reads
    ST_BKT_TILE,        // bucket path: bkt_tile_kernel
    ST_BKT_SMALL,       // bucket path: bkt_small_kernel
    ST_SP_PLAN,         // split path: windows, bitmap + ranks, tiles, descriptors, NULL rule
    ST_SP_SPLIT,        // split path: sp_split_kernel (filter + one-pass split into groups)
    ST_SP_SORT,         // split path: chunk lists per group + sp_group_kernel (sub-bin sort)
    ST_SP_TILE,         // split path: sp_tile_kernel
    ST_N
};
struct StageTimer {
    int slot;
    explicit StageTimer(int stage);
    ~StageTimer();
};

// Stream-ordered device allocation on the library stream.  Blocks of >= 16 MB are recycled by an
// exact-size cache inside the library (api.cu): every use is ordered on the single library
// stream, so handing a just-released block to the next request is safe and avoids the
// re-mapping work cudaMallocAsync does for very large blocks.
int device_alloc(void** p, size_t bytes);
void device_free(void* p);

template <class T>
inline int dalloc(T** p, size_t n) {
    *p = nullptr;
    if (n == 0) n = 1;
    return device_alloc((void**)p, n * sizeof(T));
}
template <class T>
inline void dfree(T*& p) {
    if (p) device_free((void*)p);
    p = nullptr;
}

// Several small device values -> host in ONE transfer, then a stream synchronisation: a
// one-thread kernel packs them into a device block, one copy brings the block into page-locked
// host memory.  (A cudaMemcpyAsync into pageable memory is a blocking round trip of its own, and
// the sync points of a step used to pay three of them each.)
struct FetchItem {
    const void* dev;
    void* host;
    int bytes;      // <= 32, a multiple of 4
};
int fetch_and_sync(const FetchItem* items, int n);      // n <= 8
// the same in two halves: kernels queued between them run while the host waits for the values
int fetch_begin(const FetchItem* items, int n);
int fetch_end(const FetchItem* items, int n);

// Device scratch of one call: one allocation, sub-buffers 256-byte aligned.
struct Arena {
    char* base = nullptr;
    size_t used = 0, cap = 0;
    static size_t pad(size_t bytes) { return (bytes + 255) & ~(size_t)255; }
    int reserve(size_t bytes) {
        cap = bytes;
        used = 0;
        return device_alloc(reinterpret_cast<void**>(&base), bytes > 0 ? bytes : 1);
    }
    template <class T>
    T* take(size_t n) {
        T* p = reinterpret_cast<T*>(base + used);
        used += pad(n * sizeof(T));
        return p;
    }
    ~Arena() {
        if (base) device_free(base);
    }
};

// A caller array that must be readable on the device: either the caller's own device pointer or
// a stream-ordered staging copy of host memory.
template <class T>
struct DevIn {
    const T* ptr = nullptr;
    T* owned = nullptr;
    int init(const T* src, size_t n, int mem) {
        if (mem == RCP_MEM_DEVICE || src == nullptr) {
            ptr = src;
            return RCP_OK;
        }
        RCP_TRY(dalloc(&owned, n));
        RCP_CUDA(cudaMemcpyAsync(owned, src, n * sizeof(T), cudaMemcpyHostToDevice, g_ctx.stream));
        ptr = owned;
        return RCP_OK;
    }
    ~DevIn() { dfree(owned); }
};

// ------------------------------------------------------------------ host inflate -----------
// One compressed block of a file: in_len bytes at data + in_off inflate to at most out_cap bytes
// at out + out_off; out_len receives the inflated size.
struct InflateJob {
    int64_t in_off = 0, in_len = 0, out_off = 0;
    uint32_t out_cap = 0, out_len = 0;
    uint32_t crc = 0;       // INFLATE_RAW_CRC: the CRC32 of the out_cap inflated bytes
};
enum {
    INFLATE_RAW_CRC = 0,    // raw deflate that fills out_cap exactly, CRC32 checked (BGZF)
    INFLATE_ZLIB = 1,       // zlib stream of at most out_cap bytes (bigWig data blocks)
    INFLATE_COPY = 2        // stored bytes, copied (bigWig files written uncompressed)
};
// Runs the jobs on n_threads host threads (0: one per core).  Returns -1 when every job
// succeeded, -2 when zlib could not be initialised, else the index of a failed job.
int64_t inflate_jobs(const uint8_t* data, InflateJob* jobs, int64_t n_jobs, uint8_t* out, int n_threads,
                     int kind);

// ------------------------------------------------------------------ reads index ------------
// Strand classes of the sorted arrays.  ALL is used when no strand restriction applies.
enum { CLS_ALL = 0, CLS_PLUS = 1, CLS_MINUS = 2, CLS_STAR = 3, CLS_N = 4 };

struct SortedClass {
    bool built = false;       // xs and ye (or the uniform-width stand-ins) sorted
    bool xs_sorted = false;   // xs alone is sorted (enough for the GRangesList path)
    int64_t n = 0;
    uint32_t* xs = nullptr;   // sorted global start coordinates
    uint32_t* ye = nullptr;   // sorted global (end + 1) coordinates, sorted independently;
                              // nullptr in uniform-width mode (ye[i] == xs[i] + uniform_w)
    // uniform-width mode only: correction source for the reads whose width differs from w
    int64_t cn = 0;
    uint32_t* cxs = nullptr;  // sorted (start + w): cancels the assumed end event
    uint32_t* cye = nullptr;  // sorted true (end + 1)
};

struct ReadsIdx {
    int64_t n = 0;
    int n_chrom = 0;
    bool has_strand = false;
    uint32_t max_width = 0;             // widest read (after extension and trimming)
    uint32_t uniform_w = 0;             // > 0: reads are this wide (ye == xs + w) except n_exc
    int64_t n_exc = 0;                  // reads of another width (uniform-width mode)
    uint32_t* exc_xw = nullptr;         // their start + w, true end + 1 and strand (unsorted)
    uint32_t* exc_e1 = nullptr;
    int8_t* exc_st = nullptr;
    int key_bits = 32;
    std::vector<int64_t> chrom_len;     // host copies
    std::vector<uint32_t> chrom_off;    // n_chrom + 1, global coordinate of position 0
    int64_t* d_chrom_len = nullptr;
    uint32_t* d_chrom_off = nullptr;
    // Unknown (NA) seqlengths, passed as chrom_len <= 0: coverage(reads)[[chr]] then ends at the
    // largest end among the reads that overlap the region (coverage.R:201), so a window is NULL
    // unless a read reaches its last position.  chrom_len holds a stand-in (the largest read end of
    // the chromosome, fragment extension included) that lays the chromosomes out; the rule itself
    // is applied to the finished coverage (coverage_na_rule).
    bool any_na = false;
    std::vector<uint8_t> len_na;        // n_chrom
    uint8_t* d_len_na = nullptr;
    // raw reads in global coordinates (kept for lazily built classes / pairs)
    uint32_t* g_start = nullptr;
    uint32_t* g_end1 = nullptr;         // end + 1
    int8_t* d_strand = nullptr;         // nullptr when !has_strand
    SortedClass cls[CLS_N];
    // start-sorted pairs (lazy; RNA / GRangesList path)
    bool pairs_built = false;
    uint32_t* p_end1 = nullptr;         // (end+1) in start-sorted order
    int8_t* p_strand = nullptr;         // strand in start-sorted order (nullptr when !has_strand)
    uint32_t* p_maxend1 = nullptr;      // running max of p_end1
    size_t device_bytes = 0;
    // Binned index: EVERY read as a packed candidate word, sorted by 1-kb bin of the genome (the
    // split path run with the mask "everything").  Built by the first GRangesList call of the
    // handle (coverageRnaRef makes three coverage calls on it) and reused by every later call.
    char* bn_base = nullptr;            // owner of the three arrays below
    uint32_t* bn_cand = nullptr;
    uint32_t* bn_boff = nullptr;
    uint32_t* bn_cb = nullptr;
    int bn_P = 0;
    bool bn_stranded = false;           // the words carry the strand class
    // reads too wide for the packed word (unspliced / long reads) are kept OUT of the binned
    // index, start-sorted with the running maximum of their ends (a few per cent at most)
    int64_t ln_n = 0;
    uint32_t bn_max_pack_w = 0;         // widest read the words hold
    uint32_t* ln_xs = nullptr;          // sorted global starts
    uint32_t* ln_e1 = nullptr;          // end + 1 in that order
    int8_t* ln_st = nullptr;            // strand in that order (nullptr: all '*')
    uint32_t* ln_maxe1 = nullptr;       // running maximum of ln_e1
    // Deferred validation (rcp_set_deferred_validation): rcp_reads_load returned without waiting
    // for the map kernel; its status words are still on the device and are read by the first
    // call that uses the handle (reads_resolve, or the split path's own plan fetch).
    bool pending = false;
    bool pd_rle = false;
    unsigned int* pd_err = nullptr;
    unsigned long long* pd_cnt = nullptr;
    unsigned int* pd_w = nullptr;
    uint32_t* pd_run_total = nullptr;   // owner: pd_run_first
    uint32_t* pd_run_first = nullptr;
    uint32_t pd_exc_cap = 0;
    bool pd_eager_index = false;
    // a deferred load whose validation failed: the handle keeps its error (code and message) and
    // every later call that uses it reports that error again (its fields were never filled in)
    int failed = RCP_OK;
    std::string failed_msg;
    unsigned int h_err = 0, h_w[4] = {0, 0, 0, 0}, h_total = 0;   // h_w: exceptions, width, reads wider than long_thr
    // reads wider than the packed candidate word of the split path (counted by the map kernel, so
    // that the handle's long-read list needs no counting pass and no host synchronisation)
    uint32_t long_thr = 0;
    int64_t n_long = 0;
    unsigned long long h_cnt[4] = {0, 0, 0, 0};
};

// Split path geometry: position bits of a candidate word for a genome of `span` global positions
// (<= 1024 groups of 2^P positions, 16 <= P <= 22).
inline int split_position_bits(int64_t span) {
    int P = 16;
    while (P < 22 && ((span + (1ll << P) - 1) >> P) > 1024) P++;
    return P;
}

// deferred validation: the fetch items of a pending handle (appended), and what follows the fetch.
// reads_finish and reads_resolve return the error of a failed validation on every call after it too.
int reads_pending_items(ReadsIdx& r, FetchItem* items, int* n);
int reads_finish(ReadsIdx& r);
int reads_resolve(ReadsIdx& r);     // fetch + finish when pending

int reads_build_class(ReadsIdx& r, int cls);   // lazily build a strand class
int reads_build_pairs(ReadsIdx& r);            // lazily build the start-sorted pair arrays
void reads_release(ReadsIdx& r);

// ------------------------------------------------------------------ coverage ---------------
struct Coverage {
    int64_t n_regions = 0;
    int64_t total_padded = 0;    // ints allocated in `cov`
    int64_t total_len = 0;       // sum of len
    int64_t n_null = 0;
    int32_t max_len = 0;         // longest region (sizes the staging buffers of the bin kernel)
    int path = 0;                // RCP_PATH_* that produced it (0: list / concat)
    int64_t candidates = 0;      // split path: reads that passed the bitmap filter
    // split path: n_null / total_len / candidates are produced on the device after the call has
    // returned; they are fetched on first use (coverage_resolve_stats)
    unsigned long long* d_stats = nullptr;   // [0] n_null [1] total_len [2] max_len [3] candidates [4] bound
    bool stats_pending = false;
    double scale = 1.0;
    int value_type = RCP_VALUE_INT32;   // RCP_VALUE_FLOAT32: `cov` holds float bits (signal tracks)
    // Split path: d_stats + 4, the most reads any tile of the call can apply (see cov_narrow).
    // nullptr (every other path, and RCP_COVERAGE_WIDE=1): `cov` holds 4-byte words.
    const unsigned long long* d_bound = nullptr;
    int32_t* cov = nullptr;      // dense 4-byte words (2-byte when narrow), region r at [off[r], off[r] + len[r])
    int64_t* off = nullptr;      // n_regions + 1, multiples of 32 ints
    int32_t* len = nullptr;      // n_regions, 0 for NULL
    uint8_t* is_null = nullptr;  // n_regions
};
void coverage_release(Coverage& c);
int coverage_resolve_stats(Coverage& c);

// Narrow storage.  Every read adds at most 1 to any position, so no count of a tile exceeds the
// number of reads the tile applies; when that bound is <= 65 535 for every tile of a call, the
// split path stores the coverage as uint16 (same element offsets, half the bytes).  The decision
// is a device word, read by every kernel that reads the coverage: the host never waits for it.
constexpr unsigned long long NARROW_MAX = 0xffffull;
__device__ __forceinline__ bool cov_narrow(const unsigned long long* bound) {
    return bound != nullptr && *bound <= NARROW_MAX;
}
// element i of a coverage in either layout
__device__ __forceinline__ int32_t cov_at(const int32_t* cov, int64_t i, bool narrow) {
    return narrow ? (int32_t)reinterpret_cast<const uint16_t*>(cov)[i] : cov[i];
}
// NA seqlengths: regions on such chromosomes whose genomic END position nobody covers become NULL.
// end_pos == nullptr: GRanges mask (the end is the last stored position, the first on '-'
// regions); else the index of that position inside each stitched element (GRangesList masks).
int coverage_na_rule(const ReadsIdx& rd, Coverage& cv, int64_t R, const int32_t* d_chrom, const int8_t* d_strand,
                     const int64_t* d_end_pos);

ReadsIdx* get_reads(int h);
Coverage* get_coverage(int h);
int new_coverage(Coverage** out, int* handle);

// ------------------------------------------------------------------ primitives -------------
// Radix sort (sort.cu) of n keys on their bits [begin_bit, end_bit); the pair sort is stable.
// keys (and vals) must each be a whole dalloc allocation: they come back pointing at the sorted
// data, and the other buffer CUB used is freed.  n <= 1 returns at once.  Instantiated for keys
// uint32_t and unsigned long long, and for pairs uint32_t -> uint32_t, uint32_t -> int32_t and
// unsigned long long -> int32_t.
template <class K>
int sort_keys(K*& keys, int64_t n, int begin_bit, int end_bit);
template <class K, class V>
int sort_pairs(K*& keys, V*& vals, int64_t n, int begin_bit, int end_bit);
// running maximum (index.cu)
int running_max_u32_device(const uint32_t* in, uint32_t* out, int64_t n);
// exclusive prefix sum of int64 (scan.cu); out may alias in; total (optional) receives the sum
// on the DEVICE (d_total) -- nothing is synchronised.
int exclusive_scan_i64(const int64_t* in, int64_t* out, int64_t n, int64_t* d_total);
int exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* d_total);
// the same over the first min(n_upper, *n_dev) elements: the length lives on the device, the
// launch is sized for n_upper and the blocks beyond the real length return at once
int exclusive_scan_u32_bounded(const uint32_t* in, uint32_t* out, int64_t n_upper, const uint32_t* n_dev,
                               uint32_t* d_total);
// sample.int(n, k) from a running base-R stream, dispatched as base R does (api.cu); out 1-based
struct RRng;
void r_sample_int(RRng& rng, int64_t n, int64_t k, int32_t* out);
int exclusive_scan2_i64(const int64_t* in0, int64_t* out0, int64_t* d_total0, const int64_t* in1,
                        int64_t* out1, int64_t* d_total1, int64_t n);

}  // namespace rcp
