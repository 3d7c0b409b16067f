/*
 * recoup_b200.h -- plain C ABI of librecoup_b200.so
 *
 * B200-native (sm_100a) implementation of recoup's coverage -> profile-matrix hot path.
 * The reference (hjanime/recoup, /root/reference) is interpreted R with NO native interface
 * (NAMESPACE:1-33 has no useDynLib); the path sits behind exported R closures.  Each entry point
 * below names the reference closure (file:line under /root/reference) whose body it replaces.
 * The R-side binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - coordinates 1-based closed [start,end]; strand +1 '+', -1 '-', 0 '*'.
 *   - chromosomes are dense ids 0..n_chrom-1 (as.integer(seqnames)-1).
 *   - every function returns RCP_OK (0) or an RCP_ERR_* code; rcp_last_error() gives the text.
 *     Nothing longjmps / calls back into the host language.  Per-region failures of the
 *     reference ("Caught invalid genomic area!", coverage.R:217-222) are DATA (a NULL coverage),
 *     never errors.
 *   - the caller owns every pointer it passes; outputs are caller-allocated.  The library owns
 *     device memory behind integer handles (reads / coverage), released by the *_free calls or
 *     rcp_shutdown().
 *   - `mem` says where the caller's arrays live: RCP_MEM_HOST (pageable or pinned host memory)
 *     or RCP_MEM_DEVICE (pointers valid on the bound GPU; no copies are made).
 *   - one process drives one GPU (rcp_init(device)); calls are serialised by the caller.
 *   - there is NO CPU fallback: without a usable sm_100 GPU every compute call fails with
 *     RCP_ERR_NOGPU.
 */
#ifndef RECOUP_B200_H
#define RECOUP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCP_ABI_VERSION 1

enum {
    RCP_OK = 0,
    RCP_ERR_CUDA = 1,        /* a CUDA runtime call failed                      */
    RCP_ERR_ARG = 2,         /* bad argument (R's stop() in the reference)      */
    RCP_ERR_HANDLE = 3,      /* unknown / freed handle                          */
    RCP_ERR_NOGPU = 4,       /* no CUDA device, or rcp_init() not called        */
    RCP_ERR_UNSUPPORTED = 5, /* documented unsupported corner (see DESIGN.md)   */
    RCP_ERR_DATA = 6         /* input arrays violate the stated contract        */
};

#define RCP_MEM_HOST 0
#define RCP_MEM_DEVICE 1

/* `strand` argument of calcCoverage (coverage.R:126,141-144): NULL or one of "+","-","*" */
#define RCP_STRAND_ANY 2

/* `where` of binCoverageMatrix/baseCoverageMatrix (profile.R:100-101,153-155) */
#define RCP_WHERE_WHOLE 0      /* flank = NULL */
#define RCP_WHERE_CENTER 1
#define RCP_WHERE_UPSTREAM 2
#define RCP_WHERE_DOWNSTREAM 3

#define RCP_STAT_MEAN 0
#define RCP_STAT_MEDIAN 1

#define RCP_INTERP_AUTO 0
#define RCP_INTERP_SPLINE 1
#define RCP_INTERP_LINEAR 2          /* dead code in the reference (util.R:49) -> UNSUPPORTED */
#define RCP_INTERP_NEIGHBORHOOD 3

#define RCP_SAMPLE_REJECTION 0       /* R >= 3.6.0 sample.kind (default) */
#define RCP_SAMPLE_ROUNDING 1        /* R <  3.6.0                       */

/* ---------------------------------------------------------------- library / device -------- */
const char* rcp_last_error(void);
int rcp_abi_version(void);
/* Bind this process to CUDA device `device` (one process per GPU). Replaces the reference's
 * "grid launch" cmclapply (util.R:364-382): `rc` is accepted and ignored by the R shim. */
int rcp_init(int device);
int rcp_shutdown(void);
int rcp_device_info(int* device, int* sm_count, int* cc_major, int* cc_minor, int64_t* mem_bytes);
/* cudaStream_t on which every kernel of the library is launched (for external event timing). */
void* rcp_stream(void);
int rcp_sync(void);
/* Kernels launched by this library since rcp_init / the last reset (bench.py "gpu_launches"). */
int64_t rcp_launch_count(int reset);

/* Page-locked host buffers for outputs (profile matrices): device->host copies into them run at
 * full PCIe rate.  Released buffers are kept by the library and handed out again on an
 * exact-size match, so a loop over samples pays the page-locking cost once. */
int rcp_host_alloc(int64_t bytes, void** ptr_out);
int rcp_host_free(void* ptr);

/* Optional CUDA-event timing of the library's stages on its own stream (bench.py roofline).
 * rcp_timing_read synchronises, then reports accumulated milliseconds / launches per stage
 * (stage i is named rcp_timing_stage_name(i); NULL past the last stage). */
int rcp_timing_enable(int on);
int rcp_timing_read(int reset, int capacity, double* ms_out, int64_t* count_out);
const char* rcp_timing_stage_name(int stage);

/* How rcp_coverage (GRanges masks) finds the reads of each region.  All give identical results.
 *   RCP_PATH_SPLIT    ONE streaming pass over the unsorted reads: a block bitmap of the mask in
 *                     shared memory filters them, the survivors are packed into 32-bit words and
 *                     split into <= 1024 groups of the mask's blocks through shared-memory rings
 *                     (64-byte chunks, no histogram pass, no prefix sum over the reads); each
 *                     group is then sorted by 2-kb sub-bin and every output tile reads the
 *                     sub-bins under it.  The host synchronises once, right after the plan.
 *                     Needs reads narrower than the packed word allows (<= 8191 bp, less for
 *                     dense masks / stranded calls); otherwise the call uses the paths below;
 *   RCP_PATH_BUCKETS  two passes over the unsorted reads drop each read into the buckets of the
 *                     output tiles it overlaps (cell table + hit list, no sort);
 *   RCP_PATH_INDEX    the reads are radix-sorted once per handle and every region is served by
 *                     rank searches (cheaper when one handle serves many masks);
 *   RCP_PATH_AUTO     (default) the index when the handle already has one; else split when the
 *                     reads fit its packed word; else buckets, which hand the call to the index
 *                     when the mask is dense and the reads many;
 *   RCP_PATH_BLOCKS   retired value: still accepted, selects RCP_PATH_BUCKETS (no coverage
 *                     reports it).
 * The reference has one path (findOverlaps per region, coverage.R:189-193); this is a tuning
 * knob with no counterpart there. */
#define RCP_PATH_AUTO 0
#define RCP_PATH_INDEX 1
#define RCP_PATH_BUCKETS 2
#define RCP_PATH_BLOCKS 3
#define RCP_PATH_SPLIT 4
int rcp_set_coverage_path(int path);
/* Which path produced a coverage (RCP_PATH_SPLIT / BUCKETS / INDEX; 0 for GRangesList and
 * concatenated coverages) and, for the split path, how many reads passed its bitmap filter
 * (bench.py derives that path's algorithmic bytes from it). */
int rcp_coverage_path_info(int cov, int* path, int64_t* candidates);

/* Deferred validation of the reads (default off).  When on, rcp_reads_load* return as soon as
 * their work is enqueued -- no host synchronisation -- and a data error of the reads (bad
 * chromosome id, start < 1, ...) is reported by the FIRST call that uses the reads handle
 * (rcp_coverage, rcp_coverage_list) instead of by the load itself.  Host arrays passed to a
 * deferred load must stay unchanged until that call returns.  The reference validates inside
 * GRanges construction; which call raises is the only difference.  A handle that failed its
 * validation keeps the error: every later call that uses it (rcp_coverage*, rcp_coverage_list,
 * rcp_coverage_profile) returns the same code and message; rcp_reads_info and rcp_reads_free work. */
int rcp_set_deferred_validation(int on);

/* ---------------------------------------------------------------- base-R RNG -------------- */
/* `set.seed(seed); sample(1:n, k)` -- the bin layout of splitVector (util.R:78-79). */
int rcp_r_sample(int n, int k, int seed, int sample_kind, int* out /* k */);
/* rank[i] = position (1-based) of bin i+1 in `set.seed(seed); sample(1:n, n)`; bin i gets an
 * extra base iff rank[i] <= dif (util.R:74-80). */
int rcp_r_rank_table(int n, int seed, int sample_kind, int* rank_out /* n */);

/* ---------------------------------------------------------------- reads ------------------- */
/* Upload decoded reads (the `ranges` GRanges produced by preprocessRanges, ranges.R:1-65),
 * validate them and map them to global coordinates on the device (the sorted index is built
 * lazily by the first call that needs it).  `strand` may be NULL (all '*').
 * chrom_len[c] is the seqlength; <= 0 means unknown (R's NA): coverage(reads)[[chr]] then ends at
 * the largest end among the reads that overlap a region (coverage.R:201), i.e. a window on such a
 * chromosome is NULL unless a read reaches its last position (the load then takes one extra pass
 * over the reads and one host synchronisation).  Reads must satisfy 1 <= start <= end and, after
 * the optional extension, are trimmed into [1, chrom_len] like readBam's trim() (ranges.R:117;
 * nothing to trim at on a chromosome of unknown length).  frag_len > 0 applies the fragment extension named by the north star
 * (`trim(resize(reads, frag_len, fix="start"))`; absent from the reference snapshot), 0 = off. */
int rcp_reads_load(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                   const int8_t* strand, int n_chrom, const int64_t* chrom_len, int frag_len,
                   int mem, int* reads_out);
/* The same with the chromosome ids as runs -- the form a GRanges holds them in (`seqnames(x)` is
 * a factor-Rle: run_chrom = as.integer(runValue(seqnames(x))) - 1L, run_len = runLength(...));
 * coordinate-sorted reads have one run per chromosome, so 4 of the 13 bytes per read never cross
 * PCIe.  The run lengths must be >= 0 and sum to n (< 2^32).  Same result as rcp_reads_load on the
 * expanded ids. */
int rcp_reads_load_rle(int64_t n, int64_t n_runs, const int32_t* run_chrom, const int32_t* run_len,
                       const int32_t* start, const int32_t* end, const int8_t* strand, int n_chrom,
                       const int64_t* chrom_len, int frag_len, int mem, int* reads_out);
/* The same for a library whose reads all have ONE width -- fixed-length single-end reads, or a
 * GRanges after `resize(x, w)`: an IRanges holds (start, width), and a constant width is one number
 * (`w <- width(x)[1L]` when `S4Vectors::isConstant(width(x))`, checked once at import).  Every read
 * is [start, start + width - 1]; the `end` array never crosses PCIe (9 -> 5 bytes per read with the
 * seqnames as runs).  chrom == NULL: the seqnames come as runs (n_runs, run_chrom, run_len, as in
 * rcp_reads_load_rle); otherwise dense ids and the run arguments are ignored.  Same result as
 * rcp_reads_load with end = start + width - 1. */
int rcp_reads_load_width(int64_t n, const int32_t* chrom, int64_t n_runs, const int32_t* run_chrom,
                         const int32_t* run_len, const int32_t* start, int width, const int8_t* strand,
                         int n_chrom, const int64_t* chrom_len, int frag_len, int mem, int* reads_out);
/* The read-import step right before the path (preprocessRanges / readBam, ranges.R:1-65,
 * 111-134), for reads that are already decoded (SURVEY 8f N3):
 *
 * rcp_reads_width_quantile  quantile(width(reads), prob), type 7 -- the cut of spliceAction =
 *   "remove" (ranges.R:126-127) -- and how many reads are not wider than it (the library size
 *   that "downsample" / "sampleto" then draw from).
 * rcp_r_sample_sorted  set.seed(seed) ONCE, then sort(sample(n[c], k[c])) for c = 0..n_calls-1
 *   from the one RNG stream, as the lapply over samples does (ranges.R:38-41, 55-58); sample()
 *   dispatches like base R's sample.int: the hash variant (redraw duplicates, at most 100
 *   tries) when n > 1e7 and k <= n/2, else the partial Fisher-Yates loop.  Serial by nature
 *   (one Mersenne-Twister stream): host code.  out = the blocks one after the other, 1-based.
 * rcp_reads_load_select  reads[-which(width > max_width)][idx] (ranges.R:128-130 then 43,62) and
 *   rcp_reads_load of the result, the selection done on the device.  max_width < 0: no width
 *   filter; idx NULL: keep every surviving read, else k 1-based positions among the SURVIVING
 *   reads in their original order.  *n_kept_out = reads that survive the width filter. */
int rcp_reads_width_quantile(int64_t n, const int32_t* start, const int32_t* end, double prob, int mem,
                             double* quantile_out /* host */, int64_t* n_le_out /* host */);
int rcp_r_sample_sorted(int seed, int sample_kind, int n_calls, const int64_t* n, const int64_t* k,
                        int32_t* out /* host, sum(k) */);
int rcp_reads_load_select(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                          const int8_t* strand, double max_width, int64_t k, const int32_t* idx,
                          int n_chrom, const int64_t* chrom_len, int frag_len, int mem,
                          int64_t* n_kept_out, int* reads_out);
/* The decode itself (readBam / readBed, ranges.R:111-146; SURVEY 8f N3), on the device.  The
 * result is a `decoded` handle: chrom id, start, end (1-based, closed), strand (+1 / -1 / 0) in
 * FILE ORDER, resident in HBM.
 *
 * rcp_bam_index   walks the length-prefixed alignment records of an INFLATED BAM (the bytes after
 *   the header and the reference list, e.g. from rcp_bgzf_inflate): *n_records_out
 *   = records; offsets_out (may be NULL; capacity >= records + 1) = byte offset of every record
 *   and of the end.  Host code: the chain is serial.
 * rcp_bam_decode  readGAlignments(file) with its default flag filter (unmapped records dropped),
 *   then as(., "GRanges") (splice_split = 0: one range per alignment, start = pos + 1, width =
 *   the CIGAR's extent on the reference, M D N = X) or unlist(grglist(.)) (splice_split = 1,
 *   spliceAction "split": the runs of M D = X between N operations, empty ones dropped), strand
 *   from flag 0x10, then trim() against ref_len.  rec / offsets: host or device memory (`mem`);
 *   ref_len: host, the header's reference lengths.
 * rcp_bed_decode  import.bed(file, trackLine = FALSE): lines of chrom, chromStart, chromEnd
 *   [, name, score, strand] separated by tabs or blanks; start = chromStart + 1; strand '.' or
 *   absent = '*'; empty lines, '#' comments, "track" and "browser" lines skipped.  names: the
 *   seqlevels (host), chrom id = index into them; a name not among them is RCP_ERR_DATA.
 * rcp_decoded_fetch  the arrays -> host (any pointer may be NULL).
 * rcp_reads_load_decoded  rcp_reads_load of the decoded reads without a host round trip. */
/* BGZF, the container of a BAM file (SAMv1 4.1): gzip members of <= 64 KB that carry their own
 * compressed size, inflated independently by n_threads host threads (0: one per core; zlib).
 * rcp_bgzf_size: inflated bytes and blocks of the file; rcp_bgzf_inflate: the inflated bytes (the
 * BAM header, then the alignment records).  Host code, no GPU needed; RCP_ERR_DATA when the data
 * is not BGZF (e.g. plain gzip) or a block fails its CRC32 / ISIZE. */
int rcp_bgzf_size(const uint8_t* data /* host */, int64_t n_bytes, int64_t* inflated_bytes, int64_t* n_blocks);
int rcp_bgzf_inflate(const uint8_t* data /* host */, int64_t n_bytes, uint8_t* out /* host */, int64_t capacity,
                     int n_threads);
int rcp_bam_index(const uint8_t* rec /* host */, int64_t n_bytes, int64_t* n_records_out,
                  int64_t* offsets_out /* host */, int64_t capacity);
int rcp_bam_decode(const uint8_t* rec, int64_t n_bytes, const int64_t* offsets, int64_t n_records,
                   int n_ref, const int64_t* ref_len /* host */, int splice_split, int mem,
                   int* decoded_out, int64_t* n_out);
/* rcp_bam_decode_param  rcp_bam_decode under a ScanBamParam (readGAlignments(file, param =
 *   bamParams), Rsamtools / GenomicAlignments documented behaviour).  The filters act on each
 *   record before its ranges are made; trim(), split and the caller's "remove" act on what passes.
 *   Every mapped record is checked for errors, whether the filters keep it or not.
 *   flag       (host) {keep0, keep1} = bamFlag(param, asInteger = TRUE) over the 12 flag bits
 *              0x1 .. 0x800; NULL = no flag filter.  A record passes iff every bit set in FLAG is
 *              set in keep1 and every bit clear in FLAG is set in keep0 (scanBamFlag: TRUE clears
 *              the bit in keep0, FALSE in keep1, NA leaves both).  Unmapped records (0x4) are
 *              dropped whatever the flag words say, as readGAlignments ANDs isUnmappedQuery = FALSE.
 *   mapq_min   keep MAPQ >= mapq_min (255 "unavailable" is the number 255); < 0: no filter (NA).
 *   simple_cigar  != 0: keep only a CIGAR of one M operation (10M5M is not simple).
 *   which      n_which ranges (host arrays): reference id (into the header's references), start,
 *              end, 1-based closed, 1 <= start <= end <= 536870912, in the order of
 *              as(which, "IntegerRangesList").  A record overlaps [s, e] iff POS < e and
 *              POS + span > s - 1 (POS 0-based; span = the CIGAR's M D N = X, 1 when that is 0,
 *              htslib bam_endpos), before trim().  The output is range by range, each in file
 *              order; a record that overlaps k ranges appears k times (each appearance split at
 *              its N operations under splice_split).  Needs the records sorted by (refID, POS),
 *              unplaced ones (refID -1) last -- checked on the records, RCP_ERR_DATA if not.
 *              n_which = 0: no which, file order, unsorted records are fine.
 *   tagFilter  n_tags (<= 32) tags, tag_names = their 2 characters one after the other; tag k
 *              accepts the values [tag_ptr[k], tag_ptr[k+1]) of int_values (tag_type[k] = 0,
 *              matches the integer fields c C s S i I by value) or of str_values (tag_type[k] = 1,
 *              matches Z and A fields exactly).  A record passes iff every tag is present (first
 *              occurrence) with an accepted value; a missing tag or one of another type (f, H, B,
 *              or the other kind) fails.  The aux fields after read_name, CIGAR, seq ((l_seq+1)/2
 *              bytes) and qual (l_seq bytes) are walked over every SAMv1 4.2.4 type; a field that
 *              runs past its record is RCP_ERR_DATA.  The values take at most 32 KB.
 *   With no filter given (flag NULL, mapq_min < 0, simple_cigar 0, n_which 0, n_tags 0) the
 *   result equals rcp_bam_decode's. */
int rcp_bam_decode_param(const uint8_t* rec, int64_t n_bytes, const int64_t* offsets, int64_t n_records,
                         int n_ref, const int64_t* ref_len /* host */, int splice_split, int mem,
                         const int32_t* flag /* keep0, keep1 */, int mapq_min /* < 0: NA */, int simple_cigar,
                         int n_which, const int32_t* which_ref, const int32_t* which_start,
                         const int32_t* which_end, int n_tags, const char* tag_names, const int32_t* tag_ptr,
                         const int32_t* tag_type /* 0 integer, 1 string */, const int64_t* int_values,
                         const char* const* str_values, int* decoded_out, int64_t* n_out);
int rcp_bed_decode(const char* text, int64_t n_bytes, int n_names, const char* const* names /* host */,
                   int mem, int* decoded_out, int64_t* n_out);
int rcp_decoded_fetch(int decoded, int32_t* chrom, int32_t* start, int32_t* end, int8_t* strand,
                      int64_t capacity);
int rcp_decoded_free(int decoded);
int rcp_reads_load_decoded(int decoded, int n_chrom, const int64_t* chrom_len, int frag_len,
                           int* reads_out);
/* rcp_reads_width_quantile / rcp_reads_load_select on a decoded handle (idx: host memory). */
int rcp_decoded_width_quantile(int decoded, double prob, double* quantile_out, int64_t* n_le_out);
int rcp_reads_load_decoded_select(int decoded, double max_width, int64_t k, const int32_t* idx /* host */,
                                  int n_chrom, const int64_t* chrom_len, int frag_len,
                                  int64_t* n_kept_out, int* reads_out);
int rcp_reads_info(int reads, int64_t* n, int* n_chrom, int64_t* device_bytes);
int rcp_reads_free(int reads);

/* ---------------------------------------------------------------- coverage ---------------- */
/* calcCoverage(input, mask = GRanges, strand, ignore.strand) (coverage.R:126-174 with
 * coverageFromRanges, coverage.R:176-226): one window per region, exact integer per-base
 * coverage, reversed on '-' regions, NULL when no read overlaps / window leaves the chromosome.
 * strand_filter: RCP_STRAND_ANY or +1/-1/0.  The result stays on the device behind *cov_out. */
int rcp_coverage(int reads, int64_t n_regions, const int32_t* chrom, const int32_t* start,
                 const int32_t* end, const int8_t* strand, int ignore_strand, int strand_filter,
                 int mem, int* cov_out);
/* calcCoverage(input, mask = GRangesList, ...) (coverage.R:177-178,202-207): element g owns
 * ranges ptr[g]..ptr[g+1]-1 (the exons of one gene, list order); coverage is stitched in list
 * order; chromosome and strand are those of the element's FIRST range (coverage.R:182,185);
 * a read overlapping k ranges of the element counts k times (coverage.R:190-192). */
int rcp_coverage_list(int reads, int64_t n_elements, const int64_t* ptr, const int32_t* chrom,
                      const int32_t* start, const int32_t* end, const int8_t* strand,
                      int ignore_strand, int strand_filter, int mem, int* cov_out);
/* The merge step of coverageRnaRef (coverage.R:115-120): c(left, center, right) per element,
 * NULL if any part is NULL. */
int rcp_coverage_concat3(int left, int center, int right, int* cov_out);
/* Linear normalisation (recoup.R:559-577): every coverage value is multiplied by `factor`. */
int rcp_coverage_set_scale(int cov, double factor);
int rcp_coverage_info(int cov, int64_t* n_regions, int64_t* total_len, int64_t* n_null,
                      double* scale);
/* lengths(coverage): 0 for NULL entries (profile.R:6). */
int rcp_coverage_lengths(int cov, int32_t* len_out /* n_regions */);
/* Copy the unscaled integer coverage of regions [first, first+count) to the host, packed back to
 * back (region i occupies len[i] ints).  `capacity` = ints available in `out`. */
int rcp_coverage_fetch(int cov, int64_t first, int64_t count, int32_t* out, int64_t capacity);
/* The same regions as integer run-length encodings -- the Rle objects calcCoverage returns
 * (coverage.R:171-173, contract T1 of SURVEY 8a: `input[[s]]$coverage` is a list of integer Rle
 * or NULL).  run_ptr_out (count + 1) receives the offset of each region's runs; region i owns
 * values / lengths [run_ptr[i], run_ptr[i+1]) with sum(lengths) = len[i]; NULL regions own none.
 * Call with values_out = lengths_out = NULL to size the buffers (run_ptr_out[count] = total runs),
 * then again with `capacity` entries in each.  The encoding runs on the device (run heads by
 * neighbour comparison, compaction by prefix sums): only the runs cross PCIe. */
int rcp_coverage_rle(int cov, int64_t first, int64_t count, int64_t* run_ptr_out,
                     int32_t* values_out, int32_t* lengths_out, int64_t capacity);
int rcp_coverage_free(int cov);

/* ---------------------------------------------------------------- signal tracks ----------- */
/* BigWig input (coverageFromBigWig, coverage.R:228-322: import.bw(file, as = "RleList")[[chr]]
 * subscripted by the window like the reads path).
 *
 * rcp_bigwig_load  the whole file (UCSC bbi / bigWig, little-endian) -> a `signal` handle resident
 *   in HBM.  The header and both trees are parsed on the host and the data blocks inflated there
 *   (zlib; n_threads host threads, 0 = one per core); the inflated sections are then uploaded once,
 *   expanded to items (start, end 1-based closed, float value) and validated on the device, with
 *   one host synchronisation.  RCP_ERR_DATA (the message names the block and item) when: a magic
 *   is wrong (a bigBed file says so), the file is truncated, a section's size disagrees with its
 *   item count, the items of a chromosome are not sorted and disjoint, an item leaves
 *   [1, chromSize], or a value is NaN or infinite.  A big-endian file is RCP_ERR_UNSUPPORTED.
 *   Zoom levels are skipped.  -0.0 is stored as +0.0.
 * rcp_signal_info    chromosomes, items, and the bytes rcp_signal_chroms needs for the names.
 * rcp_signal_chroms  the chromosome names (NUL-terminated, back to back) and sizes, in chromId order.
 * rcp_signal_fetch   the items (host arrays, any may be NULL) in (chromosome, start) order.
 * rcp_signal_coverage  calcCoverage(<bigwig>, mask): element g owns ranges ptr[g]..ptr[g+1]-1
 *   (ptr == NULL: one range per element, a GRanges mask).  chrom = ids into the track's
 *   chromosomes, -1 = not in the track.  Per element the chromosome and strand are those of its
 *   FIRST range (coverage.R:182,185); the vector is the track's value per base (0 between items)
 *   at the element's positions in range order, reversed when that strand is '-'.  NULL when the
 *   chromosome is not in the track, a range ends past chromSize or starts below 0 (R's subscript
 *   errors), or the element has no position; a window no item overlaps is a zero vector, not
 *   NULL.  end < start - 1 is RCP_ERR_DATA.  The result is an ordinary coverage handle of value
 *   type FLOAT32.
 * rcp_coverage_value_type  RCP_VALUE_INT32 (reads) or RCP_VALUE_FLOAT32 (signal tracks).  Every
 *   consumer of a coverage handle accepts both (bins: fp64 sums of the float values; medians
 *   exact); rcp_coverage_concat3 needs one type in all three.  rcp_coverage_fetch / _rle take
 *   INT32 handles, the _f32 twins FLOAT32 handles (RCP_ERR_ARG otherwise). */
#define RCP_VALUE_INT32 0
#define RCP_VALUE_FLOAT32 1
int rcp_bigwig_load(const uint8_t* data /* host */, int64_t n_bytes, int n_threads, int* signal_out);
int rcp_signal_info(int signal, int* n_chrom, int64_t* n_items, int64_t* names_bytes);
int rcp_signal_chroms(int signal, char* names /* NUL-terminated, back to back */, int64_t* chrom_len);
int rcp_signal_fetch(int signal, int32_t* chrom, int32_t* start, int32_t* end, float* value, int64_t capacity);
int rcp_signal_free(int signal);
int rcp_signal_coverage(int signal, int64_t n_elements, const int64_t* ptr, const int32_t* chrom,
                        const int32_t* start, const int32_t* end, const int8_t* strand, int mem, int* cov_out);
int rcp_coverage_value_type(int cov, int* type);
/* rcp_coverage_storage_bytes  2 or 4: the bytes per stored element of an INT32 handle.  The split
 *   path stores uint16 counts when no tile of the call can exceed 65 535 (environment variable
 *   RCP_COVERAGE_WIDE set: always 4); fetch, RLE and every consumer see the same int32 values
 *   either way.  May synchronise the library stream. */
int rcp_coverage_storage_bytes(int cov, int* bytes);
int rcp_coverage_fetch_f32(int cov, int64_t first, int64_t count, float* out, int64_t capacity);
int rcp_coverage_rle_f32(int cov, int64_t first, int64_t count, int64_t* run_ptr_out,
                         float* values_out, int32_t* lengths_out, int64_t capacity);

/* ---------------------------------------------------------------- profile matrix ---------- */
/* binCoverageMatrix(cvrg, binSize, stat, interpolation, flank, where) (profile.R:153-212) with
 * splitVector (util.R:15-85): writes an [n_regions x n_bins] block, column-major with leading
 * dimension ld >= n_regions, at `out`.  NULL coverage -> zero row (profile.R:191-197).
 * n_bins <= 38399 (RCP_ERR_UNSUPPORTED above).  A segment shorter than n_bins is interpolated
 * (util.R:17-73), which holds at most 5569 bins: with more bins such a segment is
 * RCP_ERR_UNSUPPORTED (the matrix is then incomplete); without one, any n_bins up to 38399 works. */
int rcp_bin_matrix(int cov, int where, int f1, int f2, int n_bins, int stat, int interp,
                   int seed, int sample_kind, double* out, int64_t ld, int mem);
/* baseCoverageMatrix(cvrg, flank, where) (profile.R:100-151): [n_regions x n_cols] per-base
 * block, same layout.  RCP_WHERE_WHOLE: n_cols must equal the common region length. */
int rcp_base_matrix(int cov, int where, int f1, int f2, int64_t n_cols, double* out, int64_t ld,
                    int mem);
/* Number of columns profileMatrix produces (profile.R:13-96) for these parameters. */
int rcp_profile_ncols(int cov, int equal_lengths, int f1, int f2, int flank_bin_size,
                      int region_bin_size, int64_t* ncols_out);
/* profileMatrix for ONE sample (profile.R:1-98): `equal_lengths` is the decision the reference
 * takes on the first sample (profile.R:6-10).  Writes cbind(left, center, right). */
int rcp_profile_matrix(int cov, int equal_lengths, int f1, int f2, int flank_bin_size,
                       int region_bin_size, int stat, int interp, int seed, int sample_kind,
                       double* out, int64_t ld, int mem);

/* ---------------------------------------------------------------- fused path -------------- */
/* coverageRef + profileMatrix (mean) for fixed-width windows (coverage.R:1-42 + profile.R:83-96):
 * windows of equal length (else RCP_ERR_ARG), n_bins bins (0 = per base), the matrix scaled by
 * `scale`.  With n_bins >= 1, windows at least n_bins long and reads the split path accepts, the
 * coverage is NEVER materialised: the tile kernel adds each tile's bin sums to 64-bit
 * accumulators and a last kernel divides -- same integer sums, same fp64 divide, so the matrix
 * equals rcp_coverage + rcp_profile_matrix bit for bit.  Otherwise the two stages are composed
 * and the coverage is released at once.  is_null_out (n_regions, may be NULL) receives the NULL
 * flags. */
int rcp_coverage_profile(int reads, int64_t n_regions, const int32_t* chrom,
                         const int32_t* start, const int32_t* end, const int8_t* strand,
                         int ignore_strand, int strand_filter, int n_bins, int seed,
                         int sample_kind, double scale, double* out, int64_t ld,
                         uint8_t* is_null_out, int mem);

/* ---------------------------------------------------------------- diagnostics ------------- */
/* Sort n 32-bit keys whose values are < 2^key_bits with the library's index sort (in place).
 * Exposed so that the index sort can be tested against a host sort. */
int rcp_sort_keys_u32(uint32_t* keys, int64_t n, int key_bits, int mem);

/* ---------------------------------------------------------------- matrix consumers -------- */
/* The reductions recoup's plotting side runs over a finished `$profile` (SURVEY 8f N4), on the
 * matrix where rcp_profile_matrix left it: column-major n_rows x n_cols, leading dimension ld,
 * `mem` says where m AND the outputs live (rcp_matrix_quantile's probs/out are always host).
 *
 * rcp_matrix_col_profile: the average curve and its band of calcPlotProfiles (plot.R:949-990):
 *   center = apply(x, 2, mean)   spread = apply(x, 2, sd)     (stat = RCP_STAT_MEAN)
 *   center = apply(x, 2, median) spread = apply(x, 2, mad)    (stat = RCP_STAT_MEDIAN; mad's
 *   constant 1.4826); log2_scale != 0 first maps x <- log2(x + 1) (plot.R:953-956).  The caller
 *   forms upper/lower = center +- spread.  sd of a single row is NaN (R: NA).
 * rcp_matrix_row_stat: apply(x, 1, sum | max | mean), the ordering values of orderProfiles
 *   (plot.R:1076-1081, 1110-1131, 1135-1146; the max variant's sample() among tied maxima
 *   returns the same value whichever it picks).  Sums and means are the correctly rounded exact
 *   value in all but pathological rows (double-double accumulation).  Non-finite cells: a sum or
 *   mean is NaN if a cell is NaN or the row holds both +Inf and -Inf, otherwise +-Inf if a cell
 *   is infinite; a finite row whose running double sum (column order) overflows gives that
 *   infinity -- R's long-double accumulator can return a finite value there.  The same rule holds
 *   for the column means of rcp_matrix_col_profile / rcp_matrix_group_col_profile.  max is NaN
 *   if a cell is NaN.
 * rcp_order: sort(v, decreasing, index.return=TRUE)$ix (plot.R:1038-1041,1100-1103): 1-based,
 *   ties keep their input order in both directions (R's default radix method), NaN/NA dropped:
 *   *n_out entries of ix are valid (R drops them: na.last = NA).
 * rcp_matrix_quantile: quantile(x, probs), type 7, over every cell (plot.R:519,536); a NaN
 *   anywhere is RCP_ERR_DATA like R's error without na.rm.  The arithmetic is quantile.default's,
 *   each operation rounded on its own: index = 1 + (n - 1) * p, lo = floor(index),
 *   h = index - lo, (1 - h) * x[lo] + h * x[hi] (1-based), R's operations in R's order; the same
 *   holds for rcp_reads_width_quantile. */
#define RCP_ROW_SUM 0
#define RCP_ROW_MAX 1
#define RCP_ROW_MEAN 2
int rcp_matrix_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int stat,
                           int log2_scale, int mem, double* center /* n_cols */,
                           double* spread /* n_cols */);
/* rcp_matrix_group_col_profile: the same curve and band per group of rows, the curves of
 *   calcDesignPlotProfiles (one per design level).  Row i belongs to group codes[i], 1-based as R
 *   stores a factor (as.integer(f), or rcp_kmeans's cluster); a code <= 0 (NA_integer_ included)
 *   excludes the row; codes == NULL puts every row in group 1.  center[g + c * n_groups] and
 *   spread[g + c * n_groups] (column-major n_groups x n_cols) are exactly what
 *   rcp_matrix_col_profile returns for the rows of group g + 1; a group without rows gets NaN in
 *   both.  m, codes and both outputs live in `mem`.  Errors: RCP_ERR_ARG as rcp_matrix_col_profile,
 *   and n_groups < 1; RCP_ERR_DATA: a code greater than n_groups (found on the device);
 *   RCP_ERR_UNSUPPORTED: more than 2^31-1 cells, or n_groups * n_cols above 2^31-1.  The launches
 *   and passes over the matrix do not depend on n_groups; the matrix is copied once into group
 *   order unless there is one group and no excluded row. */
int rcp_matrix_group_col_profile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld,
                                 const int32_t* codes /* n_rows, or NULL */, int n_groups, int stat,
                                 int log2_scale, int mem, double* center /* n_groups x n_cols */,
                                 double* spread /* n_groups x n_cols */);
int rcp_matrix_row_stat(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, int what, int mem,
                        double* out /* n_rows */);
int rcp_order(const double* v, int64_t n, int decreasing, int mem, int32_t* ix /* n */, int64_t* n_out);
int rcp_matrix_quantile(const double* m, int64_t n_rows, int64_t n_cols, int64_t ld, const double* probs,
                        int k, int mem, double* out /* k, host */);

/* ---------------------------------------------------------------- k-means ----------------- */
/* rcp_kmeans: set.seed(seed); kmeans(x, centers = k, iter.max, nstart, algorithm) -- stats::kmeans
 *   as kmeansDesign calls it (util.R:140-197, recoup.R:602).  x: column-major m x p, leading
 *   dimension ld; `mem` says where x, cluster, centers, withinss and size live; totss, iter,
 *   ifault and warnings are host scalars.
 *   Draws (host, one stream): nstart == 1: x[sample.int(m, k), ]; when those rows hold a duplicate,
 *   or nstart >= 2: cn <- unique(x) (distinct rows in first-occurrence order, -0.0 == 0.0, exact
 *   comparison), then cn[sample.int(nrow(cn), k), ] per start.  All starts run on the device; the
 *   result is the first start with the strictly smallest sum(withinss), as in R.  Distances and
 *   centres use R's floating-point operations in R's order (kmeans.c, kmns.f / AS 136), so
 *   cluster, centers, size and iter equal R's; withinss and totss are summed in another order.
 *   k == 1 runs MacQueen, as kmeans does.  k <= 256 (RCP_ERR_UNSUPPORTED above).
 *   Errors: k < 1, nstart < 1, iter_max < 1, m < k, an unknown algorithm: RCP_ERR_ARG.
 *   RCP_ERR_DATA: a non-finite x ("NA/NaN/Inf in foreign function call"), fewer distinct rows than
 *   k, Hartigan-Wong with k >= m (IFAULT 3) or an empty cluster after its first assignment
 *   (IFAULT 1), in any start.
 *   ifault (the chosen start): 0, 2 (no convergence in iter_max; iter = iter_max + 1) or 4 (the
 *   Hartigan-Wong quick-transfer stage reached 50 m steps).  warnings: RCP_KMEANS_WARN_* bits of
 *   the warnings R raises across ALL starts. */
#define RCP_KMEANS_HARTIGAN_WONG 1
#define RCP_KMEANS_LLOYD 2           /* "Lloyd" and "Forgy" */
#define RCP_KMEANS_MACQUEEN 3
#define RCP_KMEANS_WARN_NOT_CONVERGED 1    /* "did not converge in %d iterations"             */
#define RCP_KMEANS_WARN_EMPTY_CLUSTER 2    /* Lloyd / MacQueen: "empty cluster: try a better
                                              set of initial centers"                        */
#define RCP_KMEANS_WARN_QUICK_TRANSFER 4   /* "Quick-TRANSfer stage steps exceeded maximum"   */
int rcp_kmeans(const double* x, int64_t m, int64_t p, int64_t ld, int k, int nstart, int iter_max,
               int algorithm, int seed, int sample_kind, int mem, int32_t* cluster /* m, 1-based */,
               double* centers /* k x p, column-major */, double* withinss /* k */, int32_t* size /* k */,
               double* totss, int* iter, int* ifault, int* warnings);
/* rcp_r_sample_int: rcp_r_sample_sorted without the sort -- set.seed(seed) once, then
 *   sample.int(n[c], k[c]) for c = 0..n_calls-1 from the one stream, in draw order (1-based). */
int rcp_r_sample_int(int seed, int sample_kind, int n_calls, const int64_t* n, const int64_t* k,
                     int32_t* out /* host, sum(k) */);

/* ---------------------------------------------------------------- hierarchical clustering - */
/* rcp_hclust: hclust(dist(x), method = "complete") -- stats::hclust of the Euclidean distances of
 *   the rows, as ComplexHeatmap clusters heat-map rows (cluster_rows = TRUE) for orderBy$what =
 *   "hc<n>" / "hca".  x: column-major n x p, leading dimension ld; `mem` says where x, merge,
 *   height and order live.  Distances use R_euclidean's floating-point operations in its order
 *   (no FMA, correctly rounded sqrt); the merges are hclust.f's (F. Murtagh, as R ships it) and
 *   merge / order are HCASS2's, so all three equal R's bit for bit:
 *     merge:  column-major (n-1) x 2; singletons -i (1-based row), clusters +s (their step);
 *             a singleton first in a mixed row, two clusters ascending;
 *     height: the n-1 merge heights;  order: the leaves left to right, 1-based.
 *   The n x n distance matrix (8 n^2 bytes) lives on the device only and is released before return.
 *   Errors: n < 2 ("must have n >= 2 objects to cluster"), n > 65536 ("size cannot be NA nor exceed
 *   65536"), p < 1 or ld < n: RCP_ERR_ARG.  A method other than RCP_HCLUST_COMPLETE:
 *   RCP_ERR_UNSUPPORTED.  A non-finite x or a distance >= 1e300 (hclust.f's INF): RCP_ERR_DATA.
 *   Too little device memory for the matrix: RCP_ERR_CUDA, naming the bytes it needs. */
#define RCP_HCLUST_COMPLETE 3      /* index in R's METHODS vector of hclust() */
int rcp_hclust(const double* x, int64_t n, int64_t p, int64_t ld, int method, int mem,
               int32_t* merge /* (n-1) x 2, column-major, R's signs */,
               double* height /* n-1 */, int32_t* order /* n, 1-based */);

/* ---------------------------------------------------------------- multi-GPU helper -------- */
/* Scatter a row block into the gathered matrix: dst[row_index[i] + c*ld_dst] =
 * src[i + c*ld_src] for i < n_rows, c < n_cols (all pointers on the device).  Used after the
 * NCCL gather of per-rank row blocks (the reference's do.call(rbind, ...), profile.R:150,208). */
int rcp_rows_scatter(const double* src, int64_t ld_src, int64_t n_rows, int64_t n_cols,
                     const int64_t* row_index, double* dst, int64_t ld_dst);

/* Place a row block into a matrix with the COPY ENGINE (one strided 2-D copy, no SM is used):
 * dst[i + c*ld_dst] = src[i + c*ld_src] for i < n_rows, c < n_cols.  `dst` may lie in another
 * GPU's memory mapped with rcp_shared_open (the block then crosses NVLink straight into its place
 * in the gathering rank's matrix -- the reference's do.call(rbind, ...), profile.R:150,208, without a
 * gather buffer or a placement pass) or in page-locked host memory.  `stream`: a cudaStream_t, or
 * NULL for the library's stream. */
int rcp_rows_put(const double* src, int64_t ld_src, int64_t n_rows, int64_t n_cols, double* dst,
                 int64_t ld_dst, void* stream);

/* Region-sharded runs (SURVEY 8e: every GPU owns a region slice plus its overlapping reads; the
 * reference's analogue is the split of the regions over mclapply workers, coverage.R:148-154,
 * each of which subsets the reads with findOverlaps).  A rank holds an arbitrary share of the
 * reads ON ITS DEVICE; spans[(r * n_chrom + c) * 2 + {0, 1}] (host) is the closed interval
 * [lo, hi] that rank r's slice covers on chromosome c (lo > hi: nothing).  A read goes to every
 * rank whose interval it overlaps; a read with a chromosome id outside [0, n_chrom) goes to rank
 * 0, whose rcp_reads_load reports it.  _count: counts_out[r] (host) = reads bound for rank r (one
 * host synchronisation).  _pack: writes them into four device arrays (chrom, start, end int32,
 * strand int8; strand / strand_out may be NULL), rank r's run starting at offsets[r] (host: the
 * exclusive prefix sum of the counts) in each -- the send buffers of the all-to-all.  The order
 * inside a run is unspecified (coverage does not depend on it). */
int rcp_reads_route_count(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end, int world,
                          int n_chrom, const int32_t* spans, int64_t* counts_out /* world, host */);
int rcp_reads_route_pack(int64_t n, const int32_t* chrom, const int32_t* start, const int32_t* end,
                         const int8_t* strand, int world, int n_chrom, const int32_t* spans,
                         const int64_t* offsets /* world, host */, int32_t* chrom_out, int32_t* start_out,
                         int32_t* end_out, int8_t* strand_out);

/* Device memory that the other processes of this box (one per GPU) can map, so that every rank's
 * rcp_profile_matrix / rcp_bin_matrix / rcp_base_matrix writes its row block STRAIGHT into the
 * matrix of the gathering rank over NVLink (out = base + first_row, ld = total rows): the
 * exchange is fused into the kernel's own stores and no gather / scatter pass runs.  The owner
 * allocates and exports a 64-byte handle (CUDA IPC), peers open it; completion is ordered by any
 * collective or barrier after the call.  rcp_shared_close undoes rcp_shared_open,
 * rcp_shared_free undoes rcp_shared_alloc. */
#define RCP_IPC_HANDLE_BYTES 64
int rcp_shared_alloc(int64_t bytes, void** ptr_out, unsigned char* handle_out /* 64 */);
int rcp_shared_open(const unsigned char* handle /* 64 */, void** ptr_out);
int rcp_shared_close(void* ptr);
int rcp_shared_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* RECOUP_B200_H */
