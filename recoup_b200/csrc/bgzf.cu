// BGZF inflate on the host (zlib): the container of a BAM file is a series of gzip members of at
// most 64 KB each, every one carrying its own compressed size in a "BC" extra field (SAMv1 section
// 4.1), so the blocks are found by a walk over the headers and inflated independently, one
// std::thread per core.  This is the file-reading step right before rcp_bam_index / rcp_bam_decode
// (readBam of the reference, /root/reference/R/ranges.R:111-134, leaves it to Rsamtools / htslib);
// no device work here -- the calls need no GPU.
#include <zlib.h>

#include <atomic>
#include <cstring>
#include <thread>
#include <vector>

#include "rcp_internal.cuh"

namespace rcp {
namespace {

struct Block {
    int64_t in_off;      // first byte of the deflate stream
    int64_t in_len;
    int64_t out_off;
    uint32_t out_len;    // ISIZE
    uint32_t crc;
};

inline uint32_t le16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
inline uint32_t le32(const uint8_t* p) { return le16(p) | (le16(p + 2) << 16); }

// walks the member headers; RCP_ERR_DATA when the data is not BGZF
int walk(const uint8_t* d, int64_t n, std::vector<Block>* blocks, int64_t* total) {
    int64_t p = 0, out = 0;
    while (p < n) {
        if (n - p < 18 || d[p] != 31 || d[p + 1] != 139 || d[p + 2] != 8 || !(d[p + 3] & 4))
            return fail(RCP_ERR_DATA, "BGZF: no gzip member with an extra field at byte %lld", (long long)p);
        const int64_t xlen = le16(d + p + 10);
        if (n - p < 12 + xlen) return fail(RCP_ERR_DATA, "BGZF: truncated extra field at byte %lld", (long long)p);
        int64_t bsize = -1;
        for (int64_t q = p + 12; q + 4 <= p + 12 + xlen;) {
            const int64_t slen = le16(d + q + 2);
            if (d[q] == 66 && d[q + 1] == 67 && slen == 2 && q + 6 <= p + 12 + xlen) bsize = (int64_t)le16(d + q + 4) + 1;
            q += 4 + slen;
        }
        if (bsize < 0) return fail(RCP_ERR_DATA, "BGZF: the member at byte %lld has no BC field (plain gzip?)", (long long)p);
        if (bsize < 12 + xlen + 8 || p + bsize > n)
            return fail(RCP_ERR_DATA, "BGZF: the block at byte %lld (size %lld) runs past the end", (long long)p, (long long)bsize);
        Block b;
        b.in_off = p + 12 + xlen;
        b.in_len = bsize - (12 + xlen) - 8;
        b.crc = le32(d + p + bsize - 8);
        b.out_len = le32(d + p + bsize - 4);
        b.out_off = out;
        if (b.out_len > 65536u) return fail(RCP_ERR_DATA, "BGZF: a block claims %u inflated bytes", b.out_len);
        out += b.out_len;
        if (blocks) blocks->push_back(b);
        p += bsize;
    }
    *total = out;
    return RCP_OK;
}

}  // namespace

// The thread pool of every host inflate (BGZF members here, bigWig data blocks in bigwig.cu):
// workers take 16 jobs at a time from a shared counter, one z_stream each.
int64_t inflate_jobs(const uint8_t* data, InflateJob* jobs, int64_t n_jobs, uint8_t* out, int n_threads,
                     int kind) {
    unsigned nt = n_threads > 0 ? (unsigned)n_threads : std::thread::hardware_concurrency();
    nt = std::max(1u, std::min<unsigned>(nt, (unsigned)std::max<int64_t>(n_jobs / 16, 1)));
    std::atomic<int64_t> next{0};
    std::atomic<int64_t> bad{-1};
    auto work = [&]() {
        z_stream z;
        memset(&z, 0, sizeof z);
        if (kind != INFLATE_COPY && inflateInit2(&z, kind == INFLATE_RAW_CRC ? -15 : 15) != Z_OK) {
            bad.store(-2);
            return;
        }
        for (;;) {
            const int64_t i0 = next.fetch_add(16);      // 16 blocks (<= 1 MB of output) at a time
            if (i0 >= n_jobs || bad.load() != -1) break;
            for (int64_t i = i0; i < std::min<int64_t>(i0 + 16, n_jobs); i++) {
                InflateJob& b = jobs[i];
                bool ok;
                if (kind == INFLATE_COPY) {
                    ok = b.in_len <= (int64_t)b.out_cap;
                    if (ok) {
                        memcpy(out + b.out_off, data + b.in_off, (size_t)b.in_len);
                        b.out_len = (uint32_t)b.in_len;
                    }
                } else {
                    inflateReset(&z);
                    z.next_in = const_cast<Bytef*>(data + b.in_off);
                    z.avail_in = (uInt)b.in_len;
                    z.next_out = out + b.out_off;
                    z.avail_out = b.out_cap;
                    if (kind == INFLATE_RAW_CRC) {
                        const int rc = b.out_cap == 0 && b.in_len <= 2 ? Z_STREAM_END : inflate(&z, Z_FINISH);
                        ok = (rc == Z_STREAM_END || (b.out_cap == 0 && rc == Z_BUF_ERROR)) && z.avail_out == 0 &&
                             (uint32_t)crc32(crc32(0L, Z_NULL, 0), out + b.out_off, b.out_cap) == b.crc;
                    } else {
                        // a zlib stream that must end within out_cap bytes
                        ok = inflate(&z, Z_FINISH) == Z_STREAM_END;
                    }
                    b.out_len = b.out_cap - z.avail_out;
                }
                if (!ok) {
                    bad.store(i);
                    break;
                }
            }
        }
        if (kind != INFLATE_COPY) inflateEnd(&z);
    };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nt; t++) pool.emplace_back(work);
    work();
    for (auto& th : pool) th.join();
    return bad.load();
}

}  // namespace rcp

using namespace rcp;

extern "C" {

int rcp_bgzf_size(const uint8_t* data, int64_t n_bytes, int64_t* inflated_bytes, int64_t* n_blocks) {
    if (n_bytes < 0 || (n_bytes > 0 && data == nullptr) || inflated_bytes == nullptr)
        return fail(RCP_ERR_ARG, "rcp_bgzf_size: bad argument");
    std::vector<Block> blocks;
    RCP_TRY(walk(data, n_bytes, &blocks, inflated_bytes));
    if (n_blocks) *n_blocks = (int64_t)blocks.size();
    return RCP_OK;
}

int rcp_bgzf_inflate(const uint8_t* data, int64_t n_bytes, uint8_t* out, int64_t capacity, int n_threads) {
    if (n_bytes < 0 || (n_bytes > 0 && data == nullptr) || capacity < 0 || (capacity > 0 && out == nullptr))
        return fail(RCP_ERR_ARG, "rcp_bgzf_inflate: bad argument");
    std::vector<Block> blocks;
    int64_t total = 0;
    RCP_TRY(walk(data, n_bytes, &blocks, &total));
    if (total > capacity)
        return fail(RCP_ERR_ARG, "rcp_bgzf_inflate: %lld inflated bytes, room for %lld", (long long)total, (long long)capacity);
    std::vector<InflateJob> jobs(blocks.size());
    for (size_t i = 0; i < blocks.size(); i++) {
        jobs[i].in_off = blocks[i].in_off;
        jobs[i].in_len = blocks[i].in_len;
        jobs[i].out_off = blocks[i].out_off;
        jobs[i].out_cap = blocks[i].out_len;
        jobs[i].crc = blocks[i].crc;
    }
    const int64_t bad = inflate_jobs(data, jobs.data(), (int64_t)jobs.size(), out, n_threads, INFLATE_RAW_CRC);
    if (bad == -2) return fail(RCP_ERR_CUDA, "rcp_bgzf_inflate: zlib could not be initialised");
    if (bad >= 0)
        return fail(RCP_ERR_DATA, "BGZF: block %lld does not inflate to its ISIZE / CRC32", (long long)bad);
    return RCP_OK;
}

}  // extern "C"
