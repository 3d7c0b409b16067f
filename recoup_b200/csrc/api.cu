// C ABI of librecoup_b200.so (include/recoup_b200.h): context, handle tables, argument checks.
#include <climits>
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>

#include "r_rng.cuh"
#include "rcp_internal.cuh"

namespace rcp {

Ctx g_ctx;
static thread_local std::string g_error;
static std::map<int, std::unique_ptr<ReadsIdx>> g_reads;
static std::map<int, std::unique_ptr<Coverage>> g_covs;
static int g_next_handle = 1;

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

// ---- device memory: stream-ordered pool + exact-size cache of large blocks ----
static const size_t kBigBlock = 16u << 20;
static const size_t kCacheLimit = 24ull << 30;
static std::map<void*, size_t> g_big_live;            // large blocks handed out
static std::multimap<size_t, void*> g_big_free;       // large blocks released, by size
static size_t g_cached_bytes = 0;

static void cache_release_all() {
    for (auto& kv : g_big_free) cudaFreeAsync(kv.second, g_ctx.stream);
    g_big_free.clear();
    g_cached_bytes = 0;
}

int device_alloc(void** p, size_t bytes) {
    *p = nullptr;
    if (bytes >= kBigBlock) {
        auto it = g_big_free.find(bytes);
        if (it != g_big_free.end()) {
            *p = it->second;
            g_cached_bytes -= bytes;
            g_big_free.erase(it);
            g_big_live[*p] = bytes;
            return RCP_OK;
        }
    }
    cudaError_t e = cudaMallocAsync(p, bytes, g_ctx.stream);
    if (e != cudaSuccess && !g_big_free.empty()) {       // give the cache back and retry once
        cudaGetLastError();
        cache_release_all();
        e = cudaMallocAsync(p, bytes, g_ctx.stream);
    }
    if (e != cudaSuccess) {
        *p = nullptr;
        return fail(RCP_ERR_CUDA, "device allocation of %zu bytes failed: %s", bytes,
                    cudaGetErrorString(e));
    }
    if (bytes >= kBigBlock) g_big_live[*p] = bytes;
    return RCP_OK;
}

void device_free(void* p) {
    if (!p) return;
    auto it = g_big_live.find(p);
    if (it != g_big_live.end()) {
        const size_t bytes = it->second;
        g_big_live.erase(it);
        if (g_cached_bytes + bytes <= kCacheLimit) {
            g_big_free.insert({bytes, p});
            g_cached_bytes += bytes;
            return;
        }
    }
    cudaFreeAsync(p, g_ctx.stream);
}

// ---- pinned host buffers with exact-size reuse ----
static std::map<void*, size_t> g_host_live;
static std::multimap<size_t, void*> g_host_free;
static size_t g_host_cached = 0;
static const size_t kHostCacheLimit = 32ull << 30;

static void host_cache_release_all() {
    for (auto& kv : g_host_free) cudaFreeHost(kv.second);
    g_host_free.clear();
    g_host_cached = 0;
}

// ---- stage timers ----
static bool g_timing = false;
struct TimerRec { int stage; cudaEvent_t a, b; };
static std::vector<TimerRec> g_pending;
static std::vector<cudaEvent_t> g_free_events;
static double g_stage_ms[ST_N];
static int64_t g_stage_count[ST_N];
static const char* const g_stage_names[ST_N] = {
    "index_map", "index_sort", "cov_plan", "cov_tile", "cov_small", "cov_list", "cov_concat",
    "prof_bin", "prof_interp", "prof_base", "fused", "bkt_plan", "bkt_count", "bkt_scatter",
    "bkt_tile", "bkt_small", "blk_filter", "blk_hist", "blk_scatter", "blk_tile", "blk_small",
    "sp_plan", "sp_split", "sp_sort", "sp_tile", "sp_small"};

static cudaEvent_t take_event() {
    if (!g_free_events.empty()) {
        cudaEvent_t e = g_free_events.back();
        g_free_events.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

StageTimer::StageTimer(int stage) : slot(-1) {
    if (!g_timing || !g_ctx.ready) return;
    TimerRec r;
    r.stage = stage;
    r.a = take_event();
    r.b = take_event();
    cudaEventRecord(r.a, g_ctx.stream);
    g_pending.push_back(r);
    slot = (int)g_pending.size() - 1;
}
StageTimer::~StageTimer() {
    if (slot >= 0 && slot < (int)g_pending.size()) cudaEventRecord(g_pending[(size_t)slot].b, g_ctx.stream);
}

static void drain_timers() {
    if (g_pending.empty()) return;
    cudaStreamSynchronize(g_ctx.stream);
    for (auto& r : g_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
            g_stage_ms[r.stage] += ms;
            g_stage_count[r.stage]++;
        }
        g_free_events.push_back(r.a);
        g_free_events.push_back(r.b);
    }
    g_pending.clear();
}

// ---- fetch_and_sync ------------------------------------------------------------------------
namespace {
struct FetchArgs {
    const uint32_t* src[8];
    int words[8];
    int n;
};
__global__ void fetch_pack_kernel(FetchArgs a, uint32_t* __restrict__ out) {
    int at = 0;
    for (int i = 0; i < a.n; i++)
        for (int k = 0; k < a.words[i]; k++) out[at++] = a.src[i][k];
}
uint32_t* g_fetch_host = nullptr;       // page-locked
}  // namespace

// fetch_begin queues the packing kernel (it writes straight into mapped page-locked host memory)
// and records an event; fetch_end waits for that event only, so kernels queued in between keep
// the GPU busy while the host wakes up and plans the next launches.
namespace {
FetchArgs g_fetch_args;
cudaEvent_t g_fetch_event = nullptr;
uint32_t* g_fetch_host_dev = nullptr;   // device-side address of g_fetch_host
}  // namespace

int fetch_begin(const FetchItem* items, int n) {
    if (n < 0 || n > 8) return fail(RCP_ERR_ARG, "internal: fetch of %d items", n);
    if (g_fetch_host == nullptr) {
        RCP_CUDA(cudaHostAlloc((void**)&g_fetch_host, 8 * 32, cudaHostAllocMapped));
        RCP_CUDA(cudaHostGetDevicePointer((void**)&g_fetch_host_dev, g_fetch_host, 0));
        RCP_CUDA(cudaEventCreateWithFlags(&g_fetch_event, cudaEventDisableTiming));
    }
    FetchArgs& a = g_fetch_args;
    a.n = n;
    for (int i = 0; i < n; i++) {
        if (items[i].bytes <= 0 || items[i].bytes > 32 || (items[i].bytes & 3))
            return fail(RCP_ERR_ARG, "internal: fetch item of %d bytes", items[i].bytes);
        a.src[i] = static_cast<const uint32_t*>(items[i].dev);
        a.words[i] = items[i].bytes / 4;
    }
    if (n > 0) {
        fetch_pack_kernel<<<1, 1, 0, g_ctx.stream>>>(a, g_fetch_host_dev);
        RCP_LAUNCHED();
    }
    RCP_CUDA(cudaEventRecord(g_fetch_event, g_ctx.stream));
    return RCP_OK;
}

int fetch_end(const FetchItem* items, int n) {
    RCP_CUDA(cudaEventSynchronize(g_fetch_event));
    int at = 0;
    for (int i = 0; i < n; i++) {
        memcpy(items[i].host, g_fetch_host + at, (size_t)items[i].bytes);
        at += g_fetch_args.words[i];
    }
    return RCP_OK;
}

int fetch_and_sync(const FetchItem* items, int n) {
    RCP_TRY(fetch_begin(items, n));
    return fetch_end(items, n);     // the event is the last thing in the stream: the stream has drained
}

int require_ready() {
    if (!g_ctx.ready)
        return fail(RCP_ERR_NOGPU, "rcp_init() has not bound a CUDA device (no CPU fallback exists)");
    return RCP_OK;
}

ReadsIdx* get_reads(int h) {
    auto it = g_reads.find(h);
    return it == g_reads.end() ? nullptr : it->second.get();
}
Coverage* get_coverage(int h) {
    auto it = g_covs.find(h);
    return it == g_covs.end() ? nullptr : it->second.get();
}
int new_coverage(Coverage** out, int* handle) {
    const int h = g_next_handle++;
    g_covs[h] = std::unique_ptr<Coverage>(new Coverage());
    *out = g_covs[h].get();
    *handle = h;
    return RCP_OK;
}
static void drop_coverage(int h) {
    auto it = g_covs.find(h);
    if (it != g_covs.end()) {
        coverage_release(*it->second);
        g_covs.erase(it);
    }
}

// implemented in the other translation units
void decoded_release_all();     // import.cu
void signal_release_all();      // bigwig.cu
int reads_load_impl(ReadsIdx& r, int64_t n, const int32_t* chrom, int64_t n_runs,
                    const int32_t* run_chrom, const int32_t* run_len, const int32_t* start,
                    const int32_t* end, const int8_t* strand, int n_chrom,
                    const int64_t* chrom_len, int frag_len, int mem, int fixed_width);
int reads_load_select_impl(ReadsIdx& r, int64_t n, const int32_t* chrom, const int32_t* start,
                           const int32_t* end, const int8_t* strand, double max_width, int64_t k,
                           const int32_t* idx, int n_chrom, const int64_t* chrom_len, int frag_len,
                           int mem, int64_t* n_kept_out);
int coverage_ranges(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                    const int32_t* end, const int8_t* strand, int ignore_strand,
                    int strand_filter, int mem, Coverage* cv);
int coverage_ranges_bucketed(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                             const int32_t* end, const int8_t* strand, int ignore_strand,
                             int strand_filter, int mem, bool may_switch, Coverage* cv);
int coverage_list(ReadsIdx& rd, int64_t G, const int64_t* ptr, const int64_t n_ranges,
                  const int32_t* chrom, const int32_t* start, const int32_t* end,
                  const int8_t* strand, int ignore_strand, int strand_filter, int mem,
                  Coverage* cv);
int coverage_ranges_blocks(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                           const int32_t* end, const int8_t* strand, int ignore_strand,
                           int strand_filter, int mem, Coverage* cv);
int coverage_ranges_split(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                          const int32_t* end, const int8_t* strand, int ignore_strand,
                          int strand_filter, int mem, Coverage* cv);
int coverage_list_split(ReadsIdx& rd, int64_t G, const int64_t* ptr, int64_t n_ranges, const int32_t* chrom,
                        const int32_t* start, const int32_t* end, const int8_t* strand, int ignore_strand,
                        int strand_filter, int mem, Coverage* cv);
int coverage_profile_split(ReadsIdx& rd, int64_t R, const int32_t* chrom, const int32_t* start,
                           const int32_t* end, const int8_t* strand, int ignore_strand,
                           int strand_filter, int mem, int n_bins, int seed, int sample_kind,
                           double scale, double* d_out, int64_t ld, uint8_t* d_is_null);
int coverage_concat3(const Coverage& a, const Coverage& b, const Coverage& c, Coverage* cv);
int coverage_fetch(const Coverage& cv, int64_t first, int64_t count, int32_t* out,
                   int64_t capacity);
int coverage_rle(const Coverage& cv, int64_t first, int64_t count, int64_t* run_ptr,
                 int32_t* values, int32_t* lengths, int64_t capacity);
int bin_matrix_device(const Coverage& cv, int where, int f1, int f2, int n_bins, int stat,
                      int interp, int seed, int sample_kind, double* d_out, int64_t ld);
int base_matrix_device(const Coverage& cv, int where, int f1, int f2, int64_t n_cols,
                       double* d_out, int64_t ld);

namespace {

// ---- region-sharded runs: which rank(s) needs a read (SURVEY 8e: "each GPU owns a region slice
// plus its overlapping reads") ----------------------------------------------------------------
constexpr int ROUTE_MAXW = 64;          // ranks
constexpr int ROUTE_CTA = 256;
constexpr int ROUTE_PER = 8;            // reads per thread: a CTA owns ROUTE_CTA * ROUTE_PER consecutive reads

// span[(r * n_chrom + c) * 2 + {0, 1}] = [lo, hi] of rank r's slice on chromosome c (lo > hi: none).
// A read with a chromosome id outside the table goes to rank 0, whose load reports it.
__device__ __forceinline__ bool route_hit(const int32_t* sp, int n_chrom, int r, int c, int s, int e) {
    if (c < 0 || c >= n_chrom) return r == 0;
    const int lo = sp[(r * n_chrom + c) * 2], hi = sp[(r * n_chrom + c) * 2 + 1];
    return e >= lo && s <= hi;
}

// PACK = false: counts[r] += reads for rank r.  PACK = true: the reads leave as four arrays (chrom,
// start, end, strand), rank r's run starting at base[r] in each; a CTA reserves its share of every run
// with one atomic per rank, so a run is written in CTA-sized contiguous pieces.
template <bool PACK>
__global__ void __launch_bounds__(ROUTE_CTA)
route_kernel(int64_t n, const int32_t* __restrict__ chrom, const int32_t* __restrict__ start,
             const int32_t* __restrict__ end, const int8_t* __restrict__ strand, int world, int n_chrom,
             const int32_t* __restrict__ span, unsigned long long* __restrict__ counts /* [world] */,
             const int64_t* __restrict__ base /* [world] */, int32_t* __restrict__ chrom_out,
             int32_t* __restrict__ start_out, int32_t* __restrict__ end_out, int8_t* __restrict__ strand_out) {
    extern __shared__ int32_t route_sp[];                   // the span table
    __shared__ unsigned int cnt[ROUTE_MAXW];
    __shared__ unsigned long long at[ROUTE_MAXW];
    for (int i = threadIdx.x; i < world * n_chrom * 2; i += ROUTE_CTA) route_sp[i] = span[i];
    if (threadIdx.x < ROUTE_MAXW) cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t first = (int64_t)blockIdx.x * (ROUTE_CTA * ROUTE_PER);
    const unsigned lane = threadIdx.x & 31;
    int c[ROUTE_PER], s[ROUTE_PER], e[ROUTE_PER];
#pragma unroll
    for (int k = 0; k < ROUTE_PER; k++) {
        const int64_t i = first + (int64_t)k * ROUTE_CTA + threadIdx.x;
        const bool in = i < n;
        c[k] = in ? chrom[i] : 0;
        s[k] = in ? start[i] : 1;
        e[k] = in ? end[i] : 0;
        if (!in) c[k] = INT_MIN;                            // beyond the reads: nowhere
    }
    // warp-uniform loops: every lane walks the same (k, r) pairs, the ballots see whole warps
    for (int r = 0; r < world; r++) {
        unsigned mine = 0;
#pragma unroll
        for (int k = 0; k < ROUTE_PER; k++)
            mine += (c[k] != INT_MIN && route_hit(route_sp, n_chrom, r, c[k], s[k], e[k])) ? 1u : 0u;
        for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
        if (lane == 0 && mine) atomicAdd(&cnt[r], mine);
    }
    __syncthreads();
    if (!PACK) {
        if ((int)threadIdx.x < world && cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)cnt[threadIdx.x]);
        return;
    }
    if ((int)threadIdx.x < world) {
        at[threadIdx.x] = (unsigned long long)base[threadIdx.x] +
                          (cnt[threadIdx.x] ? atomicAdd(&counts[threadIdx.x], (unsigned long long)cnt[threadIdx.x]) : 0ull);
        cnt[threadIdx.x] = 0;                               // now the cursor inside the CTA's piece
    }
    __syncthreads();
    for (int r = 0; r < world; r++) {
#pragma unroll
        for (int k = 0; k < ROUTE_PER; k++) {
            const bool hit = c[k] != INT_MIN && route_hit(route_sp, n_chrom, r, c[k], s[k], e[k]);
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (m == 0u) continue;
            unsigned w0 = 0;
            if (lane == 0) w0 = atomicAdd(&cnt[r], (unsigned)__popc(m));
            w0 = __shfl_sync(0xffffffffu, w0, 0);
            if (hit) {
                const unsigned long long p = at[r] + w0 + __popc(m & ((1u << lane) - 1u));
                chrom_out[p] = c[k];
                start_out[p] = s[k];
                end_out[p] = e[k];
                if (strand_out) {
                    const int64_t i = first + (int64_t)k * ROUTE_CTA + threadIdx.x;
                    strand_out[p] = strand ? strand[i] : (int8_t)0;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256)
rows_scatter_kernel(const double* __restrict__ src, int64_t ld_src, int64_t n_rows, int64_t n_cols,
                    const int64_t* __restrict__ row_index, double* __restrict__ dst,
                    int64_t ld_dst) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_rows) return;
    const int64_t c = blockIdx.y;
    dst[row_index[i] + c * ld_dst] = src[i + c * ld_src];
}

bool valid_strand_filter(int f) { return f == RCP_STRAND_ANY || f == 1 || f == -1 || f == 0; }

// Output staging: a device buffer the kernels write, copied to the caller's host matrix (column
// by column when ld differs) or the caller's own device pointer.
struct MatrixOut {
    double* dev = nullptr;
    bool owned = false;
    int64_t ld_dev = 0;
    int init(double* out, int64_t ld, int64_t rows, int64_t cols, int mem) {
        if (mem == RCP_MEM_DEVICE) {
            dev = out;
            ld_dev = ld;
            return RCP_OK;
        }
        owned = true;
        ld_dev = rows;
        return dalloc(&dev, (size_t)(rows * cols));
    }
    int finish(double* out, int64_t ld, int64_t rows, int64_t cols) {
        if (!owned) return RCP_OK;
        if (rows > 0 && cols > 0)
            RCP_CUDA(cudaMemcpy2DAsync(out, (size_t)ld * sizeof(double), dev,
                                       (size_t)ld_dev * sizeof(double),
                                       (size_t)rows * sizeof(double), (size_t)cols,
                                       cudaMemcpyDeviceToHost, g_ctx.stream));
        RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        return RCP_OK;
    }
    ~MatrixOut() {
        if (owned) dfree(dev);
    }
};

int check_bins(int n_bins, int stat, int interp) {
    if (n_bins < 1) return fail(RCP_ERR_ARG, "binSize must be >= 1 (got %d)", n_bins);
    if (stat != RCP_STAT_MEAN && stat != RCP_STAT_MEDIAN)
        return fail(RCP_ERR_ARG, "sumStat must be mean or median");
    if (interp == RCP_INTERP_LINEAR)
        return fail(RCP_ERR_UNSUPPORTED,
                    "interpolation=\"linear\" is dead code in the reference (R/util.R:49 spells "
                    "the switch label 'inear'); not reproduced");
    if (interp != RCP_INTERP_AUTO && interp != RCP_INTERP_SPLINE && interp != RCP_INTERP_NEIGHBORHOOD)
        return fail(RCP_ERR_ARG, "unknown interpolation code %d", interp);
    return RCP_OK;
}

// columns of the three blocks of profile.R:13-78 (0 = block absent)
struct Blocks {
    int64_t left, center, right;
    bool left_binned, right_binned;
};

int r_round_half_even(double x) {
    // R's round(): IEC 60559 round-half-even on the double value
    return (int)nearbyint(x);
}

int profile_blocks(const Coverage& cv, int equal_lengths, int f1, int f2, int fbs, int rbs,
                   int64_t common_len, Blocks* b) {
    b->left = b->center = b->right = 0;
    b->left_binned = b->right_binned = false;
    if (f1 < 0 || f2 < 0 || fbs < 0 || rbs < 0) return fail(RCP_ERR_ARG, "negative flank or bin size");
    if (equal_lengths) {
        b->center = rbs != 0 ? rbs : common_len;                       // profile.R:86-93
        return RCP_OK;
    }
    if (rbs < 1)
        return fail(RCP_ERR_ARG, "regionBinSize must be >= 1 when coverage lengths differ");
    b->center = rbs;
    if (fbs != 0) {                                                    // profile.R:25-57
        const double tot = (double)f1 + (double)f2;
        if (f1 != 0) {
            b->left = r_round_half_even((double)(2 * fbs) * ((double)f1 / tot));
            b->left_binned = true;
        }
        if (f2 != 0) {
            b->right = r_round_half_even((double)(2 * fbs) * ((double)f2 / tot));
            b->right_binned = true;
        }
        if ((f1 != 0 && b->left < 1) || (f2 != 0 && b->right < 1))
            return fail(RCP_ERR_ARG, "flank bin count rounds to zero");
    } else {                                                           // profile.R:58-77
        b->left = f1;
        b->right = f2;
    }
    (void)cv;
    return RCP_OK;
}

// length of the first non-NULL coverage (profile.R:103-111); synchronises.
int common_length(const Coverage& cv, int64_t* out) {
    *out = 0;
    if (cv.n_regions == 0) return RCP_OK;
    std::vector<int32_t> len((size_t)cv.n_regions);
    RCP_CUDA(cudaMemcpyAsync(len.data(), cv.len, (size_t)cv.n_regions * 4, cudaMemcpyDeviceToHost,
                             g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    for (int32_t l : len)
        if (l > 0) {
            *out = l;
            break;
        }
    return RCP_OK;
}

}  // namespace

// sample.int(n, k) as base R dispatches it: the hash variant (do_sample2: draw, redraw on a
// duplicate, at most 100 tries) when n > 1e7 and k <= n/2, else the partial Fisher-Yates loop.
void r_sample_int(RRng& rng, int64_t n, int64_t k, int32_t* out) {
    if (n > 10000000 && k <= n / 2) {
        std::vector<uint64_t> seen((size_t)((n + 63) / 64), 0);
        for (int64_t i = 0; i < k; i++) {
            uint32_t v = 0;
            for (int j = 0; j < 100; j++) {
                v = rng.index((uint32_t)n);
                if (!((seen[v >> 6] >> (v & 63)) & 1ull)) break;
            }
            seen[v >> 6] |= 1ull << (v & 63);
            out[i] = (int32_t)(v + 1);
        }
        return;
    }
    std::vector<int> x((size_t)n);
    rng.sample((int)n, (int)k, x.data(), out);
}
}  // namespace rcp

using namespace rcp;

extern "C" {

const char* rcp_last_error(void) { return g_error.c_str(); }
int rcp_abi_version(void) { return RCP_ABI_VERSION; }

int rcp_init(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(RCP_ERR_NOGPU, "no CUDA device available (%s); librecoup_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= n) return fail(RCP_ERR_ARG, "device %d outside [0, %d)", device, n);
    if (g_ctx.ready && g_ctx.device == device) return RCP_OK;
    if (g_ctx.ready) rcp_shutdown();
    RCP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RCP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(RCP_ERR_NOGPU, "device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor);
    g_ctx.device = device;
    g_ctx.sm_count = prop.multiProcessorCount;
    g_ctx.cc_major = prop.major;
    g_ctx.cc_minor = prop.minor;
    g_ctx.mem_bytes = prop.totalGlobalMem;
    RCP_CUDA(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
    // keep freed blocks in the stream-ordered pool: repeated calls reuse them without driver calls
    cudaMemPool_t pool;
    RCP_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t threshold = UINT64_MAX;
    RCP_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
    g_ctx.launches = 0;
    g_ctx.ready = true;
    return RCP_OK;
}

int rcp_shutdown(void) {
    if (!g_ctx.ready) return RCP_OK;
    for (auto& kv : g_reads) reads_release(*kv.second);
    g_reads.clear();
    for (auto& kv : g_covs) coverage_release(*kv.second);
    g_covs.clear();
    decoded_release_all();
    signal_release_all();
    cache_release_all();
    g_big_live.clear();
    host_cache_release_all();
    drain_timers();
    g_timing = false;
    for (cudaEvent_t e : g_free_events) cudaEventDestroy(e);
    g_free_events.clear();
    cudaStreamSynchronize(g_ctx.stream);
    if (g_fetch_host) cudaFreeHost(g_fetch_host);
    if (g_fetch_event) cudaEventDestroy(g_fetch_event);
    g_fetch_host = g_fetch_host_dev = nullptr;
    g_fetch_event = nullptr;
    cudaStreamDestroy(g_ctx.stream);
    g_ctx = Ctx();
    return RCP_OK;
}

int rcp_device_info(int* device, int* sm_count, int* cc_major, int* cc_minor, int64_t* mem_bytes) {
    RCP_TRY(require_ready());
    if (device) *device = g_ctx.device;
    if (sm_count) *sm_count = g_ctx.sm_count;
    if (cc_major) *cc_major = g_ctx.cc_major;
    if (cc_minor) *cc_minor = g_ctx.cc_minor;
    if (mem_bytes) *mem_bytes = (int64_t)g_ctx.mem_bytes;
    return RCP_OK;
}

void* rcp_stream(void) { return g_ctx.ready ? (void*)g_ctx.stream : nullptr; }

int rcp_sync(void) {
    RCP_TRY(require_ready());
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return RCP_OK;
}

int rcp_host_alloc(int64_t bytes, void** ptr_out) {
    RCP_TRY(require_ready());
    if (bytes < 0 || ptr_out == nullptr) return fail(RCP_ERR_ARG, "rcp_host_alloc: bad argument");
    const size_t b = bytes > 0 ? (size_t)bytes : 1;
    auto it = g_host_free.find(b);
    if (it != g_host_free.end()) {
        *ptr_out = it->second;
        g_host_cached -= b;
        g_host_free.erase(it);
    } else {
        cudaError_t e = cudaHostAlloc(ptr_out, b, cudaHostAllocDefault);
        if (e != cudaSuccess && !g_host_free.empty()) {
            cudaGetLastError();
            host_cache_release_all();
            e = cudaHostAlloc(ptr_out, b, cudaHostAllocDefault);
        }
        if (e != cudaSuccess)
            return fail(RCP_ERR_CUDA, "pinned host allocation of %zu bytes failed: %s", b,
                        cudaGetErrorString(e));
    }
    g_host_live[*ptr_out] = b;
    return RCP_OK;
}

int rcp_host_free(void* ptr) {
    if (!ptr) return RCP_OK;
    auto it = g_host_live.find(ptr);
    if (it == g_host_live.end()) return fail(RCP_ERR_HANDLE, "rcp_host_free: unknown buffer");
    const size_t b = it->second;
    g_host_live.erase(it);
    if (g_ctx.ready && g_host_cached + b <= kHostCacheLimit) {
        g_host_free.insert({b, ptr});
        g_host_cached += b;
    } else {
        cudaFreeHost(ptr);
    }
    return RCP_OK;
}

int rcp_timing_enable(int on) {
    RCP_TRY(require_ready());
    drain_timers();
    g_timing = on != 0;
    return RCP_OK;
}

int rcp_timing_read(int reset, int capacity, double* ms_out, int64_t* count_out) {
    RCP_TRY(require_ready());
    drain_timers();
    for (int i = 0; i < ST_N && i < capacity; i++) {
        if (ms_out) ms_out[i] = g_stage_ms[i];
        if (count_out) count_out[i] = g_stage_count[i];
    }
    if (reset)
        for (int i = 0; i < ST_N; i++) {
            g_stage_ms[i] = 0.0;
            g_stage_count[i] = 0;
        }
    return RCP_OK;
}

const char* rcp_timing_stage_name(int stage) {
    return (stage >= 0 && stage < ST_N) ? g_stage_names[stage] : nullptr;
}

int rcp_set_coverage_path(int path) {
    if (path != RCP_PATH_AUTO && path != RCP_PATH_INDEX && path != RCP_PATH_BUCKETS &&
        path != RCP_PATH_BLOCKS && path != RCP_PATH_SPLIT)
        return fail(RCP_ERR_ARG, "unknown coverage path %d", path);
    g_ctx.coverage_path = path;
    return RCP_OK;
}

int rcp_set_deferred_validation(int on) {
    g_ctx.deferred_validation = on != 0;
    return RCP_OK;
}

int64_t rcp_launch_count(int reset) {
    const int64_t v = g_ctx.launches;
    if (reset) g_ctx.launches = 0;
    return v;
}

// ---- RNG (host only; needs no GPU) ---------------------------------------------------------
int rcp_r_sample(int n, int k, int seed, int sample_kind, int* out) {
    if (n < 0 || k < 0 || k > n)
        return fail(RCP_ERR_ARG, "cannot take a sample of %d from a population of %d", k, n);
    if (sample_kind != RCP_SAMPLE_REJECTION && sample_kind != RCP_SAMPLE_ROUNDING)
        return fail(RCP_ERR_ARG, "unknown sample kind %d", sample_kind);
    if (k > 0 && out == nullptr) return fail(RCP_ERR_ARG, "out is NULL");
    std::vector<int> x((size_t)n);
    std::unique_ptr<RRng> rng(new RRng);
    rng->seed((uint32_t)seed, sample_kind);
    rng->sample(n, k, x.data(), out);
    return RCP_OK;
}

// set.seed(seed) once, then sample.int(n[c], k[c]) for every call from the one stream; sorted or not
static int r_sample_calls(const char* who, int seed, int sample_kind, int n_calls, const int64_t* n,
                          const int64_t* k, int32_t* out, bool sorted) {
    if (sample_kind != RCP_SAMPLE_REJECTION && sample_kind != RCP_SAMPLE_ROUNDING)
        return fail(RCP_ERR_ARG, "unknown sample kind %d", sample_kind);
    if (n_calls < 0 || (n_calls > 0 && (n == nullptr || k == nullptr)))
        return fail(RCP_ERR_ARG, "%s: bad argument", who);
    std::unique_ptr<RRng> rng(new RRng);
    rng->seed((uint32_t)seed, sample_kind);
    int64_t at = 0;
    for (int c = 0; c < n_calls; c++) {
        if (n[c] < 0 || k[c] < 0 || k[c] > n[c] || n[c] > 0x7fffffff)
            return fail(RCP_ERR_ARG, "cannot take a sample of %lld from a population of %lld",
                        (long long)k[c], (long long)n[c]);
        if (k[c] > 0 && out == nullptr) return fail(RCP_ERR_ARG, "out is NULL");
        r_sample_int(*rng, n[c], k[c], out + at);
        if (sorted) std::sort(out + at, out + at + k[c]);
        at += k[c];
    }
    return RCP_OK;
}

int rcp_r_sample_sorted(int seed, int sample_kind, int n_calls, const int64_t* n, const int64_t* k,
                        int32_t* out) {
    return r_sample_calls("rcp_r_sample_sorted", seed, sample_kind, n_calls, n, k, out, true);
}

int rcp_r_sample_int(int seed, int sample_kind, int n_calls, const int64_t* n, const int64_t* k,
                     int32_t* out) {
    return r_sample_calls("rcp_r_sample_int", seed, sample_kind, n_calls, n, k, out, false);
}

int rcp_r_rank_table(int n, int seed, int sample_kind, int* rank_out) {
    if (n < 0) return fail(RCP_ERR_ARG, "n < 0");
    std::vector<int> perm((size_t)n);
    RCP_TRY(rcp_r_sample(n, n, seed, sample_kind, perm.data()));
    for (int pos = 0; pos < n; pos++) rank_out[perm[(size_t)pos] - 1] = pos + 1;
    return RCP_OK;
}

// ---- reads ---------------------------------------------------------------------------------
int rcp_reads_load(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                   const int8_t* strand, int n_chrom, const int64_t* chrom_len, int frag_len,
                   int mem, int* reads_out) {
    RCP_TRY(require_ready());
    if (n < 0 || n_chrom < 1 || chrom_len == nullptr || reads_out == nullptr || frag_len < 0)
        return fail(RCP_ERR_ARG, "rcp_reads_load: bad scalar argument");
    if (n > 0 && (chrom == nullptr || start == nullptr || end == nullptr))
        return fail(RCP_ERR_ARG, "rcp_reads_load: NULL array");
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    std::unique_ptr<ReadsIdx> r(new ReadsIdx());
    int rc = reads_load_impl(*r, n, chrom, 0, nullptr, nullptr, start, end, strand, n_chrom, chrom_len,
                             frag_len, mem, 0);
    if (rc != RCP_OK) {
        reads_release(*r);
        return rc;
    }
    const int h = g_next_handle++;
    g_reads[h] = std::move(r);
    *reads_out = h;
    return RCP_OK;
}

int rcp_reads_load_rle(int64_t n, int64_t n_runs, const int32_t* run_chrom, const int32_t* run_len,
                       const int32_t* start, const int32_t* end, const int8_t* strand, int n_chrom,
                       const int64_t* chrom_len, int frag_len, int mem, int* reads_out) {
    RCP_TRY(require_ready());
    if (n < 0 || n_runs < 0 || n_chrom < 1 || chrom_len == nullptr || reads_out == nullptr ||
        frag_len < 0)
        return fail(RCP_ERR_ARG, "rcp_reads_load_rle: bad scalar argument");
    if (n > 0 && (n_runs < 1 || run_chrom == nullptr || run_len == nullptr || start == nullptr ||
                  end == nullptr))
        return fail(RCP_ERR_ARG, "rcp_reads_load_rle: NULL array");
    if (n >= 0xfffffff0ll) return fail(RCP_ERR_UNSUPPORTED, "rcp_reads_load_rle: n >= 2^32");
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    std::unique_ptr<ReadsIdx> r(new ReadsIdx());
    int rc = reads_load_impl(*r, n, nullptr, n_runs, run_chrom, run_len, start, end, strand, n_chrom,
                             chrom_len, frag_len, mem, 0);
    if (rc != RCP_OK) {
        reads_release(*r);
        return rc;
    }
    const int h = g_next_handle++;
    g_reads[h] = std::move(r);
    *reads_out = h;
    return RCP_OK;
}

int rcp_reads_load_width(int64_t n, const int32_t* chrom, int64_t n_runs, const int32_t* run_chrom,
                         const int32_t* run_len, const int32_t* start, int width, const int8_t* strand,
                         int n_chrom, const int64_t* chrom_len, int frag_len, int mem, int* reads_out) {
    RCP_TRY(require_ready());
    if (n < 0 || n_runs < 0 || n_chrom < 1 || chrom_len == nullptr || reads_out == nullptr || frag_len < 0)
        return fail(RCP_ERR_ARG, "rcp_reads_load_width: bad scalar argument");
    if (width < 1) return fail(RCP_ERR_ARG, "rcp_reads_load_width: width must be >= 1");
    const bool runs = chrom == nullptr;
    if (n > 0 && (start == nullptr || (runs && (n_runs < 1 || run_chrom == nullptr || run_len == nullptr))))
        return fail(RCP_ERR_ARG, "rcp_reads_load_width: NULL array");
    if (runs && n >= 0xfffffff0ll) return fail(RCP_ERR_UNSUPPORTED, "rcp_reads_load_width: n >= 2^32");
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    std::unique_ptr<ReadsIdx> r(new ReadsIdx());
    int rc = reads_load_impl(*r, n, chrom, runs ? n_runs : 0, runs ? run_chrom : nullptr,
                             runs ? run_len : nullptr, start, nullptr, strand, n_chrom, chrom_len, frag_len,
                             mem, width);
    if (rc != RCP_OK) {
        reads_release(*r);
        return rc;
    }
    const int h = g_next_handle++;
    g_reads[h] = std::move(r);
    *reads_out = h;
    return RCP_OK;
}

int rcp_reads_load_select(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                          const int8_t* strand, double max_width, int64_t k, const int32_t* idx,
                          int n_chrom, const int64_t* chrom_len, int frag_len, int mem,
                          int64_t* n_kept_out, int* reads_out) {
    RCP_TRY(require_ready());
    if (n < 0 || k < 0 || n_chrom < 1 || chrom_len == nullptr || reads_out == nullptr || frag_len < 0)
        return fail(RCP_ERR_ARG, "rcp_reads_load_select: bad scalar argument");
    if (n > 0 && (chrom == nullptr || start == nullptr || end == nullptr))
        return fail(RCP_ERR_ARG, "rcp_reads_load_select: NULL array");
    if (n >= 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "rcp_reads_load_select: n >= 2^31 - 1");
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    std::unique_ptr<ReadsIdx> r(new ReadsIdx());
    int rc = reads_load_select_impl(*r, n, chrom, start, end, strand, max_width, k, idx, n_chrom,
                                    chrom_len, frag_len, mem, n_kept_out);
    if (rc != RCP_OK) {
        reads_release(*r);
        return rc;
    }
    const int h = g_next_handle++;
    g_reads[h] = std::move(r);
    *reads_out = h;
    return RCP_OK;
}

int rcp_reads_info(int reads, int64_t* n, int* n_chrom, int64_t* device_bytes) {
    ReadsIdx* r = get_reads(reads);
    if (!r) return fail(RCP_ERR_HANDLE, "unknown reads handle %d", reads);
    if (n) *n = r->n;
    if (n_chrom) *n_chrom = r->n_chrom;
    if (device_bytes) *device_bytes = (int64_t)r->device_bytes;
    return RCP_OK;
}

int rcp_reads_free(int reads) {
    auto it = g_reads.find(reads);
    if (it == g_reads.end()) return fail(RCP_ERR_HANDLE, "unknown reads handle %d", reads);
    reads_release(*it->second);
    g_reads.erase(it);
    return RCP_OK;
}

// ---- coverage ------------------------------------------------------------------------------
int rcp_coverage(int reads, int64_t n_regions, const int32_t* chrom, const int32_t* start,
                 const int32_t* end, const int8_t* strand, int ignore_strand, int strand_filter,
                 int mem, int* cov_out) {
    RCP_TRY(require_ready());
    ReadsIdx* r = get_reads(reads);
    if (!r) return fail(RCP_ERR_HANDLE, "unknown reads handle %d", reads);
    if (n_regions < 0 || cov_out == nullptr) return fail(RCP_ERR_ARG, "rcp_coverage: bad argument");
    if (n_regions > 0 && (!chrom || !start || !end)) return fail(RCP_ERR_ARG, "rcp_coverage: NULL array");
    if (!valid_strand_filter(strand_filter)) return fail(RCP_ERR_ARG, "bad strand filter %d", strand_filter);
    if (n_regions > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 regions");
    Coverage* cv;
    int h;
    RCP_TRY(new_coverage(&cv, &h));
    // RCP_PATH_AUTO: the sorted index serves the call when it already exists (built by an
    // earlier call or by the GRangesList path); otherwise the reads are bucketed per tile, which
    // costs two passes over the reads instead of a sort.
    bool use_index = g_ctx.coverage_path == RCP_PATH_INDEX;
    if (g_ctx.coverage_path == RCP_PATH_AUTO) {
        const bool unstranded =
            (strand_filter == RCP_STRAND_ANY) && (ignore_strand != 0 || strand == nullptr);
        use_index = unstranded ? r->cls[CLS_ALL].built
                               : (r->cls[CLS_PLUS].built && r->cls[CLS_MINUS].built &&
                                  r->cls[CLS_STAR].built);
    }
    // The split path (one streaming pass over the unsorted reads) serves every GRanges mask it can
    // (reads narrower than the packed candidate word allows); it also validates a deferred load.
    int rc = RCP_SPLIT_NOT_APPLICABLE;
    const bool try_split = g_ctx.coverage_path == RCP_PATH_SPLIT ||
                           (g_ctx.coverage_path == RCP_PATH_AUTO && !use_index &&
                            getenv("RCP_AUTO_NO_SPLIT") == nullptr);
    if (try_split) {
        rc = coverage_ranges_split(*r, n_regions, chrom, start, end, strand, ignore_strand != 0,
                                   strand_filter, mem, cv);
    }
    if (rc == RCP_SPLIT_NOT_APPLICABLE) {
        rc = reads_resolve(*r);
        if (rc == RCP_OK) rc = RCP_SWITCH_TO_INDEX;
        if (rc == RCP_SWITCH_TO_INDEX && g_ctx.coverage_path == RCP_PATH_BLOCKS) {
            rc = coverage_ranges_blocks(*r, n_regions, chrom, start, end, strand, ignore_strand != 0,
                                        strand_filter, mem, cv);
        } else if (rc == RCP_SWITCH_TO_INDEX && !use_index) {
            rc = coverage_ranges_bucketed(*r, n_regions, chrom, start, end, strand, ignore_strand != 0,
                                          strand_filter, mem,
                                          g_ctx.coverage_path == RCP_PATH_AUTO ||
                                              g_ctx.coverage_path == RCP_PATH_SPLIT, cv);
            if (rc == RCP_SWITCH_TO_INDEX) coverage_release(*cv);      // dense mask, very many reads
        }
        if (rc == RCP_SWITCH_TO_INDEX)
            rc = coverage_ranges(*r, n_regions, chrom, start, end, strand, ignore_strand != 0,
                                 strand_filter, mem, cv);
    }
    if (rc == RCP_OK && r->any_na && n_regions > 0) {      // NA seqlengths: the rule of coverage.R:201
        DevIn<int32_t> d_chrom;
        DevIn<int8_t> d_strand;
        rc = d_chrom.init(chrom, (size_t)n_regions, mem);
        if (rc == RCP_OK) rc = d_strand.init(strand, (size_t)n_regions, mem);
        if (rc == RCP_OK) rc = coverage_na_rule(*r, *cv, n_regions, d_chrom.ptr, d_strand.ptr, nullptr);
    }
    if (rc != RCP_OK) {
        drop_coverage(h);
        return rc;
    }
    *cov_out = h;
    return RCP_OK;
}

int rcp_coverage_list(int reads, int64_t n_elements, const int64_t* ptr, const int32_t* chrom,
                      const int32_t* start, const int32_t* end, const int8_t* strand,
                      int ignore_strand, int strand_filter, int mem, int* cov_out) {
    RCP_TRY(require_ready());
    ReadsIdx* r = get_reads(reads);
    if (!r) return fail(RCP_ERR_HANDLE, "unknown reads handle %d", reads);
    if (n_elements < 0 || ptr == nullptr || cov_out == nullptr)
        return fail(RCP_ERR_ARG, "rcp_coverage_list: bad argument");
    if (mem != RCP_MEM_HOST)
        return fail(RCP_ERR_UNSUPPORTED, "rcp_coverage_list takes host arrays (ptr is read on the host)");
    if (!valid_strand_filter(strand_filter)) return fail(RCP_ERR_ARG, "bad strand filter %d", strand_filter);
    for (int64_t g = 0; g < n_elements; g++)
        if (ptr[g + 1] < ptr[g]) return fail(RCP_ERR_ARG, "ptr is not non-decreasing at %lld", (long long)g);
    if (ptr[0] != 0) return fail(RCP_ERR_ARG, "ptr[0] must be 0");
    const int64_t n_ranges = ptr[n_elements];
    if (n_ranges > 0 && (!chrom || !start || !end)) return fail(RCP_ERR_ARG, "rcp_coverage_list: NULL array");
    RCP_TRY(reads_resolve(*r));
    Coverage* cv;
    int h;
    RCP_TRY(new_coverage(&cv, &h));
    // the handle's binned index (built on first use) serves the call when the reads fit its packed
    // word; the start-sorted pairs (one radix sort of every read) otherwise or on request
    int rc = RCP_SPLIT_NOT_APPLICABLE;
    if ((g_ctx.coverage_path == RCP_PATH_AUTO || g_ctx.coverage_path == RCP_PATH_SPLIT) && !r->pairs_built &&
        getenv("RCP_AUTO_NO_SPLIT") == nullptr) {
        rc = coverage_list_split(*r, n_elements, ptr, n_ranges, chrom, start, end, strand, ignore_strand != 0,
                                 strand_filter, mem, cv);
        if (rc == RCP_SPLIT_NOT_APPLICABLE) coverage_release(*cv);
    }
    if (rc == RCP_SPLIT_NOT_APPLICABLE)
        rc = coverage_list(*r, n_elements, ptr, n_ranges, chrom, start, end, strand,
                           ignore_strand != 0, strand_filter, mem, cv);
    if (rc == RCP_OK && r->any_na && n_elements > 0) {
        // NA seqlengths: where the largest range end of an element sits inside its stitched vector
        // (ranges in list order, a start of 0 dropped, the whole vector reversed when the FIRST
        // range is on '-': coverage.R:185,202-215)
        std::vector<int32_t> e_chrom((size_t)n_elements, 0);
        std::vector<int8_t> e_strand((size_t)n_elements, 0);
        std::vector<int64_t> e_pos((size_t)n_elements, -1);
        for (int64_t g = 0; g < n_elements; g++) {
            const int64_t a = ptr[g], b = ptr[g + 1];
            if (b <= a) continue;
            e_chrom[(size_t)g] = chrom[a];
            e_strand[(size_t)g] = strand ? strand[a] : (int8_t)0;
            int64_t total = 0, best_end = INT64_MIN, best_pos = -1;
            for (int64_t j = a; j < b; j++) {
                const int64_t w = (int64_t)end[j] - std::max<int64_t>(start[j], 1) + 1;
                if (w <= 0) continue;
                if ((int64_t)end[j] > best_end) {
                    best_end = end[j];
                    best_pos = total + w - 1;
                }
                total += w;
            }
            if (best_pos >= 0) e_pos[(size_t)g] = e_strand[(size_t)g] < 0 ? total - 1 - best_pos : best_pos;
        }
        DevIn<int32_t> d_chrom;
        DevIn<int8_t> d_strand;
        DevIn<int64_t> d_pos;
        rc = d_chrom.init(e_chrom.data(), (size_t)n_elements, RCP_MEM_HOST);
        if (rc == RCP_OK) rc = d_strand.init(e_strand.data(), (size_t)n_elements, RCP_MEM_HOST);
        if (rc == RCP_OK) rc = d_pos.init(e_pos.data(), (size_t)n_elements, RCP_MEM_HOST);
        if (rc == RCP_OK) rc = coverage_na_rule(*r, *cv, n_elements, d_chrom.ptr, d_strand.ptr, d_pos.ptr);
    }
    if (rc != RCP_OK) {
        drop_coverage(h);
        return rc;
    }
    *cov_out = h;
    return RCP_OK;
}

int rcp_coverage_concat3(int left, int center, int right, int* cov_out) {
    RCP_TRY(require_ready());
    Coverage *a = get_coverage(left), *b = get_coverage(center), *c = get_coverage(right);
    if (!a || !b || !c) return fail(RCP_ERR_HANDLE, "unknown coverage handle");
    if (cov_out == nullptr) return fail(RCP_ERR_ARG, "cov_out is NULL");
    if (a->value_type != b->value_type || b->value_type != c->value_type)
        return fail(RCP_ERR_ARG, "concat3: the three coverages have different value types");
    Coverage* cv;
    int h;
    RCP_TRY(new_coverage(&cv, &h));
    cv->value_type = b->value_type;
    int rc = coverage_concat3(*a, *b, *c, cv);
    if (rc != RCP_OK) {
        drop_coverage(h);
        return rc;
    }
    cv->scale = b->scale;
    *cov_out = h;
    return RCP_OK;
}

int rcp_coverage_set_scale(int cov, double factor) {
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    cv->scale = factor;
    return RCP_OK;
}

int rcp_coverage_info(int cov, int64_t* n_regions, int64_t* total_len, int64_t* n_null,
                      double* scale) {
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (total_len || n_null) RCP_TRY(coverage_resolve_stats(*cv));
    if (n_regions) *n_regions = cv->n_regions;
    if (total_len) *total_len = cv->total_len;
    if (n_null) *n_null = cv->n_null;
    if (scale) *scale = cv->scale;
    return RCP_OK;
}

int rcp_coverage_path_info(int cov, int* path, int64_t* candidates) {
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (candidates) RCP_TRY(coverage_resolve_stats(*cv));
    if (path) *path = cv->path;
    if (candidates) *candidates = cv->candidates;
    return RCP_OK;
}

int rcp_coverage_lengths(int cov, int32_t* len_out) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (cv->n_regions == 0) return RCP_OK;
    if (!len_out) return fail(RCP_ERR_ARG, "len_out is NULL");
    RCP_CUDA(cudaMemcpyAsync(len_out, cv->len, (size_t)cv->n_regions * 4, cudaMemcpyDeviceToHost,
                             g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return RCP_OK;
}

int rcp_coverage_fetch(int cov, int64_t first, int64_t count, int32_t* out, int64_t capacity) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (cv->value_type != RCP_VALUE_INT32) return fail(RCP_ERR_ARG, "rcp_coverage_fetch: a FLOAT32 coverage (use _f32)");
    return coverage_fetch(*cv, first, count, out, capacity);
}

int rcp_coverage_fetch_f32(int cov, int64_t first, int64_t count, float* out, int64_t capacity) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (cv->value_type != RCP_VALUE_FLOAT32) return fail(RCP_ERR_ARG, "rcp_coverage_fetch_f32: an INT32 coverage");
    return coverage_fetch(*cv, first, count, reinterpret_cast<int32_t*>(out), capacity);
}

int rcp_coverage_value_type(int cov, int* type) {
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (type == nullptr) return fail(RCP_ERR_ARG, "type is NULL");
    *type = cv->value_type;
    return RCP_OK;
}

int rcp_coverage_storage_bytes(int cov, int* bytes) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (bytes == nullptr) return fail(RCP_ERR_ARG, "bytes is NULL");
    *bytes = 4;
    if (cv->d_bound) {
        unsigned long long bound = 0;
        const FetchItem items[1] = {{cv->d_bound, &bound, 8}};
        RCP_TRY(fetch_and_sync(items, 1));
        if (bound <= NARROW_MAX) *bytes = 2;
    }
    return RCP_OK;
}

int rcp_coverage_rle(int cov, int64_t first, int64_t count, int64_t* run_ptr_out,
                     int32_t* values_out, int32_t* lengths_out, int64_t capacity) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (cv->value_type != RCP_VALUE_INT32) return fail(RCP_ERR_ARG, "rcp_coverage_rle: a FLOAT32 coverage (use _f32)");
    return coverage_rle(*cv, first, count, run_ptr_out, values_out, lengths_out, capacity);
}

// float runs: -0.0 is stored as +0.0, so equal bits are equal values and the integer run
// encoding serves unchanged
int rcp_coverage_rle_f32(int cov, int64_t first, int64_t count, int64_t* run_ptr_out, float* values_out,
                         int32_t* lengths_out, int64_t capacity) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (cv->value_type != RCP_VALUE_FLOAT32) return fail(RCP_ERR_ARG, "rcp_coverage_rle_f32: an INT32 coverage");
    return coverage_rle(*cv, first, count, run_ptr_out, reinterpret_cast<int32_t*>(values_out), lengths_out,
                        capacity);
}

int rcp_coverage_free(int cov) {
    if (!get_coverage(cov)) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    drop_coverage(cov);
    return RCP_OK;
}

// ---- profile -------------------------------------------------------------------------------
int rcp_bin_matrix(int cov, int where, int f1, int f2, int n_bins, int stat, int interp, int seed,
                   int sample_kind, double* out, int64_t ld, int mem) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    RCP_TRY(check_bins(n_bins, stat, interp));
    if (where < RCP_WHERE_WHOLE || where > RCP_WHERE_DOWNSTREAM) return fail(RCP_ERR_ARG, "bad where");
    if (f1 < 0 || f2 < 0) return fail(RCP_ERR_ARG, "negative flank");
    if (ld < cv->n_regions || out == nullptr) return fail(RCP_ERR_ARG, "bad output matrix");
    MatrixOut m;
    RCP_TRY(m.init(out, ld, cv->n_regions, n_bins, mem));
    RCP_TRY(bin_matrix_device(*cv, where, f1, f2, n_bins, stat, interp, seed, sample_kind, m.dev,
                              m.ld_dev));
    return m.finish(out, ld, cv->n_regions, n_bins);
}

int rcp_base_matrix(int cov, int where, int f1, int f2, int64_t n_cols, double* out, int64_t ld,
                    int mem) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (where < RCP_WHERE_WHOLE || where > RCP_WHERE_DOWNSTREAM || where == RCP_WHERE_CENTER)
        return fail(RCP_ERR_ARG, "baseCoverageMatrix takes where = whole / upstream / downstream");
    if (f1 < 0 || f2 < 0 || n_cols < 0) return fail(RCP_ERR_ARG, "negative size");
    if (where == RCP_WHERE_UPSTREAM && n_cols != f1) return fail(RCP_ERR_ARG, "n_cols must equal flank[1]");
    if (where == RCP_WHERE_DOWNSTREAM && n_cols != f2) return fail(RCP_ERR_ARG, "n_cols must equal flank[2]");
    if (ld < cv->n_regions || out == nullptr) return fail(RCP_ERR_ARG, "bad output matrix");
    MatrixOut m;
    RCP_TRY(m.init(out, ld, cv->n_regions, n_cols, mem));
    RCP_TRY(base_matrix_device(*cv, where, f1, f2, n_cols, m.dev, m.ld_dev));
    return m.finish(out, ld, cv->n_regions, n_cols);
}

int rcp_profile_ncols(int cov, int equal_lengths, int f1, int f2, int flank_bin_size,
                      int region_bin_size, int64_t* ncols_out) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    int64_t common = 0;
    if (equal_lengths && region_bin_size == 0) RCP_TRY(common_length(*cv, &common));
    Blocks b;
    RCP_TRY(profile_blocks(*cv, equal_lengths, f1, f2, flank_bin_size, region_bin_size, common, &b));
    *ncols_out = b.left + b.center + b.right;
    return RCP_OK;
}

int rcp_profile_matrix(int cov, int equal_lengths, int f1, int f2, int flank_bin_size,
                       int region_bin_size, int stat, int interp, int seed, int sample_kind,
                       double* out, int64_t ld, int mem) {
    RCP_TRY(require_ready());
    Coverage* cv = get_coverage(cov);
    if (!cv) return fail(RCP_ERR_HANDLE, "unknown coverage handle %d", cov);
    if (ld < cv->n_regions || out == nullptr) return fail(RCP_ERR_ARG, "bad output matrix");
    int64_t common = 0;
    if (equal_lengths && region_bin_size == 0) RCP_TRY(common_length(*cv, &common));
    Blocks b;
    RCP_TRY(profile_blocks(*cv, equal_lengths, f1, f2, flank_bin_size, region_bin_size, common, &b));
    const int64_t ncols = b.left + b.center + b.right;
    const int64_t R = cv->n_regions;
    MatrixOut m;
    RCP_TRY(m.init(out, ld, R, ncols, mem));
    if (equal_lengths) {
        if (region_bin_size != 0) {
            // profile.R:88-90 does not forward `interpolation`: binCoverageMatrix's default "auto"
            RCP_TRY(check_bins(region_bin_size, stat, RCP_INTERP_AUTO));
            RCP_TRY(bin_matrix_device(*cv, RCP_WHERE_WHOLE, 0, 0, region_bin_size, stat,
                                      RCP_INTERP_AUTO, seed, sample_kind, m.dev, m.ld_dev));
        } else {
            RCP_TRY(base_matrix_device(*cv, RCP_WHERE_WHOLE, 0, 0, common, m.dev, m.ld_dev));
        }
    } else {
        RCP_TRY(check_bins((int)b.center, stat, interp));
        double* p = m.dev;
        if (b.left > 0) {
            if (b.left_binned)
                RCP_TRY(bin_matrix_device(*cv, RCP_WHERE_UPSTREAM, f1, f2, (int)b.left, stat, interp,
                                          seed, sample_kind, p, m.ld_dev));
            else
                RCP_TRY(base_matrix_device(*cv, RCP_WHERE_UPSTREAM, f1, f2, b.left, p, m.ld_dev));
            p += b.left * m.ld_dev;
        }
        RCP_TRY(bin_matrix_device(*cv, RCP_WHERE_CENTER, f1, f2, (int)b.center, stat, interp, seed,
                                  sample_kind, p, m.ld_dev));
        p += b.center * m.ld_dev;
        if (b.right > 0) {
            if (b.right_binned)
                RCP_TRY(bin_matrix_device(*cv, RCP_WHERE_DOWNSTREAM, f1, f2, (int)b.right, stat,
                                          interp, seed, sample_kind, p, m.ld_dev));
            else
                RCP_TRY(base_matrix_device(*cv, RCP_WHERE_DOWNSTREAM, f1, f2, b.right, p, m.ld_dev));
        }
    }
    return m.finish(out, ld, R, ncols);
}

// ---- fused path ----------------------------------------------------------------------------
// Equal-length windows with n_bins >= 1 bins are served by the split path's fused tile kernel (the coverage never reaches HBM).  Everything else (per-base matrices, windows
// shorter than the bin count, reads too wide for the split path) composes the two stages and
// releases the coverage at once.  Windows of different lengths are an error either way.
int rcp_coverage_profile(int reads, int64_t n_regions, const int32_t* chrom, const int32_t* start,
                         const int32_t* end, const int8_t* strand, int ignore_strand,
                         int strand_filter, int n_bins, int seed, int sample_kind, double scale,
                         double* out, int64_t ld, uint8_t* is_null_out, int mem) {
    RCP_TRY(require_ready());
    ReadsIdx* r = get_reads(reads);
    if (!r) return fail(RCP_ERR_HANDLE, "unknown reads handle %d", reads);
    if (n_regions < 0 || n_bins < 0 || out == nullptr || ld < n_regions)
        return fail(RCP_ERR_ARG, "rcp_coverage_profile: bad argument");
    if (n_regions > 0 && (!chrom || !start || !end)) return fail(RCP_ERR_ARG, "rcp_coverage_profile: NULL array");
    if (!valid_strand_filter(strand_filter)) return fail(RCP_ERR_ARG, "bad strand filter %d", strand_filter);
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "bad mem kind");
    if (n_regions > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 regions");
    const bool may_split = g_ctx.coverage_path == RCP_PATH_SPLIT ||
                           (g_ctx.coverage_path == RCP_PATH_AUTO && getenv("RCP_AUTO_NO_SPLIT") == nullptr);
    if (n_bins >= 1 && may_split && !r->any_na) {      // (NA seqlengths: the rule needs the coverage itself)
        MatrixOut m;
        RCP_TRY(m.init(out, ld, n_regions, n_bins, mem));
        uint8_t* d_null = nullptr;
        bool own_null = false;
        if (is_null_out) {
            if (mem == RCP_MEM_DEVICE) d_null = is_null_out;
            else {
                RCP_TRY(dalloc(&d_null, (size_t)n_regions));
                own_null = true;
            }
        }
        int rc = coverage_profile_split(*r, n_regions, chrom, start, end, strand, ignore_strand != 0,
                                        strand_filter, mem, n_bins, seed, sample_kind, scale, m.dev, m.ld_dev,
                                        d_null);
        if (rc == RCP_OK) {
            if (own_null && n_regions > 0) {
                cudaError_t e = cudaMemcpyAsync(is_null_out, d_null, (size_t)n_regions, cudaMemcpyDeviceToHost,
                                                g_ctx.stream);
                if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "null-flag copy failed: %s", cudaGetErrorString(e));
            }
            if (rc == RCP_OK) rc = m.finish(out, ld, n_regions, n_bins);     // synchronises for host output
        }
        if (own_null) dfree(d_null);
        if (rc != RCP_SPLIT_NOT_APPLICABLE) return rc;
    }
    int h = 0;
    RCP_TRY(rcp_coverage(reads, n_regions, chrom, start, end, strand, ignore_strand, strand_filter,
                         mem, &h));
    Coverage* cv = get_coverage(h);
    cv->scale = scale;
    int rc = RCP_OK;
    {   // one common length (profile.R:86-96 is the equal-length branch)
        std::vector<int32_t> len((size_t)n_regions);
        if (n_regions > 0) {
            cudaError_t e = cudaMemcpyAsync(len.data(), cv->len, (size_t)n_regions * 4, cudaMemcpyDeviceToHost,
                                            g_ctx.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
            if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "length copy failed: %s", cudaGetErrorString(e));
        }
        int32_t common = 0;
        for (int32_t l : len) {
            if (l == 0) continue;
            if (common == 0) common = l;
            else if (l != common) {
                rc = fail(RCP_ERR_ARG, "rcp_coverage_profile: the windows have different lengths (%d and %d); "
                                       "use rcp_coverage + rcp_profile_matrix", common, l);
                break;
            }
        }
    }
    if (rc == RCP_OK)
        rc = rcp_profile_matrix(h, 1, 0, 0, 0, n_bins, RCP_STAT_MEAN, RCP_INTERP_AUTO, seed, sample_kind, out,
                                ld, mem);
    if (rc == RCP_OK && is_null_out && n_regions > 0) {
        cudaError_t e = cudaMemcpyAsync(is_null_out, cv->is_null, (size_t)n_regions,
                                        mem == RCP_MEM_DEVICE ? cudaMemcpyDeviceToDevice
                                                              : cudaMemcpyDeviceToHost,
                                        g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "null-flag copy failed: %s", cudaGetErrorString(e));
    }
    drop_coverage(h);
    return rc;
}

int rcp_sort_keys_u32(uint32_t* keys, int64_t n, int key_bits, int mem) {
    RCP_TRY(require_ready());
    if (n < 0 || key_bits < 1 || key_bits > 32 || (n > 0 && keys == nullptr))
        return fail(RCP_ERR_ARG, "rcp_sort_keys_u32: bad argument");
    if (n == 0) return RCP_OK;
    if (mem == RCP_MEM_DEVICE) return sort_keys_u32(keys, n, key_bits);
    uint32_t* d = nullptr;
    RCP_TRY(dalloc(&d, (size_t)n));
    RCP_CUDA(cudaMemcpyAsync(d, keys, (size_t)n * 4, cudaMemcpyHostToDevice, g_ctx.stream));
    int rc = sort_keys_u32(d, n, key_bits);
    if (rc == RCP_OK) {
        cudaError_t e = cudaMemcpyAsync(keys, d, (size_t)n * 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "sort copy failed: %s", cudaGetErrorString(e));
    }
    dfree(d);
    return rc;
}

// ---- peer-mapped device memory (CUDA IPC) --------------------------------------------------
int rcp_shared_alloc(int64_t bytes, void** ptr_out, unsigned char* handle_out) {
    RCP_TRY(require_ready());
    if (bytes <= 0 || ptr_out == nullptr || handle_out == nullptr)
        return fail(RCP_ERR_ARG, "rcp_shared_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == RCP_IPC_HANDLE_BYTES, "IPC handle size");
    void* p = nullptr;
    RCP_CUDA(cudaMalloc(&p, (size_t)bytes));      // not from the stream-ordered pool: exportable
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(RCP_ERR_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    }
    memcpy(handle_out, &h, sizeof(h));
    *ptr_out = p;
    return RCP_OK;
}

int rcp_shared_open(const unsigned char* handle, void** ptr_out) {
    RCP_TRY(require_ready());
    if (handle == nullptr || ptr_out == nullptr) return fail(RCP_ERR_ARG, "rcp_shared_open: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    RCP_CUDA(cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return RCP_OK;
}

int rcp_shared_close(void* ptr) {
    if (ptr == nullptr) return RCP_OK;
    RCP_CUDA(cudaIpcCloseMemHandle(ptr));
    return RCP_OK;
}

int rcp_shared_free(void* ptr) {
    if (ptr == nullptr) return RCP_OK;
    RCP_CUDA(cudaFree(ptr));
    return RCP_OK;
}

int rcp_rows_put(const double* src, int64_t ld_src, int64_t n_rows, int64_t n_cols, double* dst,
                 int64_t ld_dst, void* stream) {
    RCP_TRY(require_ready());
    if (n_rows <= 0 || n_cols <= 0) return RCP_OK;
    if (src == nullptr || dst == nullptr || ld_src < n_rows || ld_dst < n_rows)
        return fail(RCP_ERR_ARG, "rcp_rows_put: bad argument");
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : g_ctx.stream;
    RCP_CUDA(cudaMemcpy2DAsync(dst, (size_t)ld_dst * 8, src, (size_t)ld_src * 8, (size_t)n_rows * 8, (size_t)n_cols,
                               cudaMemcpyDefault, st));
    return RCP_OK;
}

static int route_impl(bool pack, int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                      const int8_t* strand, int world, int n_chrom, const int32_t* spans, int64_t* counts_host,
                      const int64_t* offsets_host, int32_t* chrom_out, int32_t* start_out, int32_t* end_out,
                      int8_t* strand_out) {
    RCP_TRY(require_ready());
    if (n < 0 || world < 1 || world > ROUTE_MAXW || n_chrom < 1 || spans == nullptr)
        return fail(RCP_ERR_ARG, "rcp_reads_route: bad scalar argument (1 <= world <= %d)", ROUTE_MAXW);
    if (n > 0 && (!chrom || !start || !end)) return fail(RCP_ERR_ARG, "rcp_reads_route: NULL array");
    const size_t sp_ints = (size_t)world * n_chrom * 2;
    if (sp_ints * 4 > 40 * 1024) return fail(RCP_ERR_UNSUPPORTED, "rcp_reads_route: span table over 40 KB");
    int32_t* d_span = nullptr;
    unsigned long long* d_cnt = nullptr;
    int64_t* d_base = nullptr;
    RCP_TRY(dalloc(&d_span, sp_ints));
    RCP_TRY(dalloc(&d_cnt, (size_t)world));
    RCP_TRY(dalloc(&d_base, (size_t)world));
    RCP_CUDA(cudaMemcpyAsync(d_span, spans, sp_ints * 4, cudaMemcpyHostToDevice, g_ctx.stream));
    RCP_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)world * 8, g_ctx.stream));
    if (pack)
        RCP_CUDA(cudaMemcpyAsync(d_base, offsets_host, (size_t)world * 8, cudaMemcpyHostToDevice, g_ctx.stream));
    const unsigned grid = (unsigned)std::max<int64_t>(1, (n + ROUTE_CTA * ROUTE_PER - 1) / (ROUTE_CTA * ROUTE_PER));
    if (n > 0) {
        if (pack)
            route_kernel<true><<<grid, ROUTE_CTA, sp_ints * 4, g_ctx.stream>>>(n, chrom, start, end, strand, world,
                                                                             n_chrom, d_span, d_cnt, d_base, chrom_out,
                                                                             start_out, end_out, strand_out);
        else
            route_kernel<false><<<grid, ROUTE_CTA, sp_ints * 4, g_ctx.stream>>>(n, chrom, start, end, strand, world,
                                                                              n_chrom, d_span, d_cnt, nullptr,
                                                                              nullptr, nullptr, nullptr, nullptr);
        RCP_LAUNCHED();
    }
    int rc = RCP_OK;
    if (!pack) {
        RCP_CUDA(cudaMemcpyAsync(counts_host, d_cnt, (size_t)world * 8, cudaMemcpyDeviceToHost, g_ctx.stream));
        RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    }
    dfree(d_span);
    dfree(d_cnt);
    dfree(d_base);
    return rc;
}

int rcp_reads_route_count(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end, int world,
                          int n_chrom, const int32_t* spans, int64_t* counts_out) {
    if (counts_out == nullptr) return fail(RCP_ERR_ARG, "rcp_reads_route_count: counts_out is NULL");
    return route_impl(false, n, chrom, start, end, nullptr, world, n_chrom, spans, counts_out, nullptr, nullptr,
                      nullptr, nullptr, nullptr);
}

int rcp_reads_route_pack(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                         const int8_t* strand, int world, int n_chrom, const int32_t* spans,
                         const int64_t* offsets, int32_t* chrom_out, int32_t* start_out, int32_t* end_out,
                         int8_t* strand_out) {
    if (offsets == nullptr || (n > 0 && (chrom_out == nullptr || start_out == nullptr || end_out == nullptr)))
        return fail(RCP_ERR_ARG, "rcp_reads_route_pack: NULL argument");
    return route_impl(true, n, chrom, start, end, strand, world, n_chrom, spans, nullptr, offsets, chrom_out,
                      start_out, end_out, strand_out);
}

int rcp_rows_scatter(const double* src, int64_t ld_src, int64_t n_rows, int64_t n_cols,
                     const int64_t* row_index, double* dst, int64_t ld_dst) {
    RCP_TRY(require_ready());
    if (n_rows <= 0 || n_cols <= 0) return RCP_OK;
    if (n_cols > 65535) return fail(RCP_ERR_UNSUPPORTED, "rows_scatter: more than 65535 columns");
    rows_scatter_kernel<<<dim3((unsigned)((n_rows + 255) / 256), (unsigned)n_cols), 256, 0,
                          g_ctx.stream>>>(src, ld_src, n_rows, n_cols, row_index, dst, ld_dst);
    RCP_LAUNCHED();
    return RCP_OK;
}

}  // extern "C"
