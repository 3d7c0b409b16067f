// Device radix sorts of the library: CUB's DeviceRadixSort (toolkit header templates), one pass
// per 8-bit digit.  Every radix sort goes through the two functions here: the index (sorted
// starts and ends, start-sorted (start, read id) pairs), the long-read list of the binned index,
// the matrix consumers (orderings, quantiles, row groups) and k-means (distinct rows).  Only the
// segmented sort of the group medians (consumers.cu) calls CUB itself.
//
// The sorts hand back whichever buffer CUB finished in (declared in rcp_internal.cuh), so no
// sorted array is copied back.  They are instantiated at the end of this file for the types in
// use, which keeps the CUB header out of the other translation units.
#include <cub/device/device_radix_sort.cuh>

#include <type_traits>
#include <utility>

#include "rcp_internal.cuh"

namespace rcp {

namespace {

// a device buffer of one sort, freed on every return path
template <class T>
struct Scratch {
    T* p = nullptr;
    ~Scratch() { dfree(p); }
};

}  // namespace

template <class K>
int sort_keys(K*& keys, int64_t n, int begin_bit, int end_bit) {
    if (n <= 1) return RCP_OK;
    // 32-bit keys are the index's read coordinates
    if (sizeof(K) == 4 && n > 0x3fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^30-1 reads in one sort");
    if (n > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 values in one sort");
    Scratch<K> alt;
    Scratch<uint8_t> tmp;
    RCP_TRY(dalloc(&alt.p, (size_t)n));
    cub::DoubleBuffer<K> kb(keys, alt.p);
    size_t tmp_bytes = 0;
    RCP_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, kb, (int)n, begin_bit, end_bit, g_ctx.stream));
    RCP_TRY(dalloc(&tmp.p, tmp_bytes));
    RCP_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, kb, (int)n, begin_bit, end_bit, g_ctx.stream));
    g_ctx.launches += 1 + (end_bit - begin_bit + 7) / 8;
    if (kb.Current() != keys) std::swap(keys, alt.p);
    return RCP_OK;
}

template <class K, class V>
int sort_pairs(K*& keys, V*& vals, int64_t n, int begin_bit, int end_bit) {
    if (n <= 1) return RCP_OK;
    // uint32_t values are read ids (the index), int32_t ones rows or cells (the matrix consumers)
    if (n > 0x7fffffff)
        return fail(RCP_ERR_UNSUPPORTED, "more than 2^31-1 %s in one sort",
                    std::is_same<V, uint32_t>::value ? "reads" : "values");
    Scratch<K> kalt;
    Scratch<V> valt;
    Scratch<uint8_t> tmp;
    RCP_TRY(dalloc(&kalt.p, (size_t)n));
    RCP_TRY(dalloc(&valt.p, (size_t)n));
    cub::DoubleBuffer<K> kb(keys, kalt.p);
    cub::DoubleBuffer<V> vb(vals, valt.p);
    size_t tmp_bytes = 0;
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, kb, vb, (int)n, begin_bit, end_bit,
                                             g_ctx.stream));
    RCP_TRY(dalloc(&tmp.p, tmp_bytes));
    RCP_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, kb, vb, (int)n, begin_bit, end_bit,
                                             g_ctx.stream));
    g_ctx.launches += 1 + (end_bit - begin_bit + 7) / 8;
    if (kb.Current() != keys) std::swap(keys, kalt.p);
    if (vb.Current() != vals) std::swap(vals, valt.p);
    return RCP_OK;
}

template int sort_keys<uint32_t>(uint32_t*&, int64_t, int, int);
template int sort_keys<unsigned long long>(unsigned long long*&, int64_t, int, int);
template int sort_pairs<uint32_t, uint32_t>(uint32_t*&, uint32_t*&, int64_t, int, int);
template int sort_pairs<uint32_t, int32_t>(uint32_t*&, int32_t*&, int64_t, int, int);
template int sort_pairs<unsigned long long, int32_t>(unsigned long long*&, int32_t*&, int64_t, int, int);

}  // namespace rcp
