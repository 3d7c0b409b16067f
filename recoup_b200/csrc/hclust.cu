// hclust(dist(x), method = "complete") of stats, the row clustering ComplexHeatmap applies to a heat
// map (cluster_rows = TRUE) when orderBy$what is "hc<n>" / "hca", on the device.
//
// Parity with R's own arithmetic is the goal, as for k-means: every distance is R_euclidean's
// `dev = x[i,c] - x[j,c]; d += dev * dev` over the columns in order, then sqrt, with explicit
// __d*_rn intrinsics (the file is also built with -fmad=false).  The merge sequence is F.
// Murtagh's hclust.f as R ships it, complete linkage, restated literally: the nearest neighbour
// (NN / DISNN) of every row among the rows to its right, the alive row with the strictly smallest
// DISNN giving the pair (lowest index on ties), d(I2, k) = max(d(I2, k), d(J2, k)), the new NN of
// I2, the `k < I2` branch, and the rescan of every row whose NN was I2 or J2.
//
//   * hc_dist_kernel: a SYRK-shaped tiling on the fp64 CUDA cores.  A CTA owns a 64 x 64 tile of
//     pairs with tile row <= tile column, stages both row tiles of x through shared memory one
//     16-column chunk at a time (so each pair still sums its columns in order) and gives each
//     thread a 4 x 4 register block of pairs.  The tile goes back through shared memory so that
//     both triangles of the full n x n matrix are stored with coalesced rows.  Tensor cores are of
//     no use: |a|^2 + |b|^2 - 2 a.b is not R's arithmetic.
//   * hc_nn_kernel: one warp per row, the initial NN to the right (lowest index on ties).
//   * hc_merge_kernel: all n - 1 merges in one launch of ONE thread-block cluster.  CTA r owns a
//     contiguous slice of rows and keeps their DISNN / NN in its shared memory, next to a private
//     copy of the alive flags of every row (every CTA learns J2 at the same time).  Per merge:
//       1. each CTA's argmin over its alive rows, published in its shared memory; cluster barrier;
//          every CTA reads the others' candidates (distributed shared memory) and takes the same
//          pair;
//       2. each CTA updates row I2 and column I2 of the matrix for the k of its slice, keeps its
//          best k > I2 as a candidate for the new NN of I2 and applies the k < I2 branch;
//       3. each CTA rescans its rows whose NN was I2 or J2, all its threads on one row at a
//          time; cluster barrier;
//       4. the owner of I2 takes the new NN of I2 from the candidates.
//     The matrix is streamed from L2 / HBM with L1-bypassing loads and stores: a row is read by
//     whichever CTA owns the column, and the cluster barrier (release / acquire at cluster scope)
//     orders those accesses between steps.
//   * merge and order (HCASS2) are built on the host in O(n) from IA / IB.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "rcp_internal.cuh"

namespace cg = cooperative_groups;

namespace rcp {
namespace {

constexpr int TPB = 256;
constexpr int DT = 64;                  // pairs tile: DT x DT
constexpr int DK = 16;                  // columns staged per chunk
constexpr int MERGE_THREADS = 1024;
constexpr double HC_INF = 1e300;        // hclust.f's INF
constexpr int64_t HC_MAX_N = 65536;     // R's limit of hclust()
constexpr int NO_ROW = 0x7fffffff;

__global__ void __launch_bounds__(TPB)
hc_finite_kernel(const double* __restrict__ x, int64_t n, int64_t p, int64_t ld, int* __restrict__ bad) {
    const int64_t tot = n * p;
    for (int64_t t = (int64_t)blockIdx.x * TPB + threadIdx.x; t < tot; t += (int64_t)gridDim.x * TPB) {
        const int64_t j = t / n, i = t - j * n;
        if (!isfinite(x[i + j * ld])) {
            *bad = 1;
            return;
        }
    }
}

// Tile t of the upper triangle of tiles (tile row bi <= tile column bj), column by column.
__device__ __forceinline__ void tile_of(int64_t t, int* bi, int* bj) {
    int j = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
    while ((int64_t)(j + 1) * (j + 2) / 2 <= t) j++;
    while ((int64_t)j * (j + 1) / 2 > t) j--;
    *bj = j;
    *bi = (int)(t - (int64_t)j * (j + 1) / 2);
}

// D (n x n, row-major, leading dimension n) = dist(x); *big = 1 when a distance is >= INF.
__global__ void __launch_bounds__(TPB)
hc_dist_kernel(const double* __restrict__ x, int n, int64_t p, int64_t ld, double* __restrict__ D,
               int* __restrict__ big) {
    // the staged chunks and, after the last chunk, the finished tile share one buffer
    __shared__ double buf[DT * (DT + 1)];
    double(*As)[DT] = reinterpret_cast<double(*)[DT]>(buf);
    double(*Bs)[DT] = reinterpret_cast<double(*)[DT]>(buf + DK * DT);
    double(*Ts)[DT + 1] = reinterpret_cast<double(*)[DT + 1]>(buf);
    int bi, bj;
    tile_of(blockIdx.x, &bi, &bj);
    const int i0 = bi * DT, j0 = bj * DT;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
    for (int64_t c0 = 0; c0 < p; c0 += DK) {
        const int kc = p - c0 < DK ? (int)(p - c0) : DK;
        for (int e = threadIdx.x; e < DK * DT; e += TPB) {
            const int c = e / DT, r = e - c * DT;
            double a = 0.0, b = 0.0;
            if (c < kc) {
                if (i0 + r < n) a = x[(i0 + r) + (c0 + c) * ld];
                if (j0 + r < n) b = x[(j0 + r) + (c0 + c) * ld];
            }
            As[c][r] = a;
            Bs[c][r] = b;
        }
        __syncthreads();
        for (int c = 0; c < kc; c++) {
            double av[4], bv[4];
#pragma unroll
            for (int a = 0; a < 4; a++) av[a] = As[c][ty + 16 * a];
#pragma unroll
            for (int b = 0; b < 4; b++) bv[b] = Bs[c][tx + 16 * b];
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const double dev = __dsub_rn(av[a], bv[b]);
                    acc[a][b] = __dadd_rn(acc[a][b], __dmul_rn(dev, dev));
                }
        }
        __syncthreads();
    }
    bool over = false;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const double d = __dsqrt_rn(acc[a][b]);
            const int i = i0 + ty + 16 * a, j = j0 + tx + 16 * b;
            if (i < n && j < n && i != j && d >= HC_INF) over = true;
            Ts[ty + 16 * a][tx + 16 * b] = d;
        }
    if (over) *big = 1;
    __syncthreads();
    // rows i0.. (row-major tile) and the mirror rows j0.. (the tile transposed), coalesced
    for (int e = threadIdx.x; e < DT * DT; e += TPB) {
        const int r = e / DT, c = e - r * DT;
        if (i0 + r < n && j0 + c < n) D[(int64_t)(i0 + r) * n + j0 + c] = Ts[r][c];
        if (j0 + r < n && i0 + c < n) D[(int64_t)(j0 + r) * n + i0 + c] = Ts[c][r];
    }
}

// (d, i) < (e, j): the smaller distance, then the lower index
__device__ __forceinline__ bool before(double d, int i, double e, int j) { return d < e || (d == e && i < j); }

__device__ __forceinline__ void warp_argmin(double& d, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double e = __shfl_xor_sync(0xffffffffu, d, o);
        const int j = __shfl_xor_sync(0xffffffffu, i, o);
        if (before(e, j, d, i)) {
            d = e;
            i = j;
        }
    }
}

// the argmin of the CTA's (d, i) pairs, returned to every thread; red holds 32 pairs
__device__ __forceinline__ void block_argmin(double& d, int& i, double* red_d, int* red_i) {
    warp_argmin(d, i);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        red_d[w] = d;
        red_i[w] = i;
    }
    __syncthreads();
    if (w == 0) {
        const int nw = blockDim.x >> 5;
        d = lane < nw ? red_d[lane] : HC_INF;
        i = lane < nw ? red_i[lane] : NO_ROW;
        warp_argmin(d, i);
        if (lane == 0) {
            red_d[32] = d;
            red_i[32] = i;
        }
    }
    __syncthreads();
    d = red_d[32];
    i = red_i[32];
    __syncthreads();
}

// The initial NN of row i: the row j > i with the strictly smallest distance (lowest index on
// ties), over a warp; (INF, -1) for the last row.
__device__ __forceinline__ void warp_row_nn(const double* __restrict__ D, int n, int i, double& dmin, int& jmin) {
    const int lane = threadIdx.x & 31;
    dmin = HC_INF;
    jmin = NO_ROW;
    const double* row = D + (int64_t)i * n;
    for (int j = i + 1 + lane; j < n; j += 32) {
        const double v = __ldcg(row + j);
        if (v < dmin) {
            dmin = v;
            jmin = j;
        }
    }
    warp_argmin(dmin, jmin);
    if (jmin == NO_ROW) jmin = -1;
}

__global__ void __launch_bounds__(TPB)
hc_nn_kernel(const double* __restrict__ D, int n, double* __restrict__ disnn, int* __restrict__ nn) {
    const int i = (int)(((int64_t)blockIdx.x * TPB + threadIdx.x) >> 5);
    if (i >= n) return;
    double d;
    int j;
    warp_row_nn(D, n, i, d, j);
    if ((threadIdx.x & 31) == 0) {
        disnn[i] = d;
        nn[i] = j;
    }
}

struct Cand {
    double d;
    int i, j;
};

// All n - 1 merges of hclust.f (complete linkage) in one cluster of gridDim.x CTAs; CTA r owns rows
// [r * S, min(n, (r + 1) * S)).  Dynamic shared memory: alive[n] (padded), disnn[S], nn[S], list[S].
__global__ void __launch_bounds__(MERGE_THREADS, 1)
hc_merge_kernel(double* __restrict__ D, int n, int S, const double* __restrict__ disnn0,
                const int* __restrict__ nn0, int* __restrict__ ia, int* __restrict__ ib, double* __restrict__ crit) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ double red_d[33];
    __shared__ int red_i[33];
    __shared__ Cand cand;           // this CTA's best row (phase 1)
    __shared__ Cand nnc;            // this CTA's best k > I2 (phase 2)
    __shared__ int s_pair[2];
    __shared__ int n_list;
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int npad = (n + 15) & ~15;
    unsigned char* alive = smem;
    double* disnn = reinterpret_cast<double*>(smem + npad);
    int* nn = reinterpret_cast<int*>(disnn + S);
    int* list = nn + S;
    const int r0 = min(n, rank * S), r1 = min(n, r0 + S);
    const int tid = threadIdx.x, nt = blockDim.x;

    for (int k = tid; k < n; k += nt) alive[k] = 1;
    for (int r = r0 + tid; r < r1; r += nt) {
        disnn[r - r0] = r < n - 1 ? disnn0[r] : HC_INF;
        nn[r - r0] = r < n - 1 ? nn0[r] : -1;
    }
    __syncthreads();

    for (int step = 0; step < n - 1; step++) {
        // 1. the pair: the alive row with the strictly smallest DISNN, lowest index on ties
        double d = HC_INF;
        int im = NO_ROW;
        for (int r = r0 + tid; r < r1; r += nt)
            if (alive[r] && before(disnn[r - r0], r, d, im)) {
                d = disnn[r - r0];
                im = r;
            }
        block_argmin(d, im, red_d, red_i);
        if (tid == 0) cand = Cand{d, im, im == NO_ROW ? -1 : nn[im - r0]};
        cluster.sync();
        if (tid == 0) {
            Cand best{HC_INF, NO_ROW, -1};
            for (int q = 0; q < C; q++) {
                const Cand c = *cluster.map_shared_rank(&cand, q);
                if (c.d < HC_INF && before(c.d, c.i, best.d, best.i)) best = c;
            }
            const int I2 = min(best.i, best.j), J2 = max(best.i, best.j);
            s_pair[0] = I2;
            s_pair[1] = J2;
            alive[J2] = 0;
            if (rank == 0) {
                ia[step] = I2;
                ib[step] = J2;
                crit[step] = best.d;
            }
        }
        __syncthreads();
        const int I2 = s_pair[0], J2 = s_pair[1];

        // 2. d(I2, k) = max(d(I2, k), d(J2, k)) for the alive k != I2 of this slice
        double* rowI = D + (int64_t)I2 * n;
        const double* rowJ = D + (int64_t)J2 * n;
        d = HC_INF;
        int kb = NO_ROW;
        for (int k = r0 + tid; k < r1; k += nt) {
            if (!alive[k] || k == I2) continue;
            const double v = fmax(__ldcg(rowI + k), __ldcg(rowJ + k));
            __stcg(rowI + k, v);
            __stcg(D + (int64_t)k * n + I2, v);
            if (I2 < k) {
                if (v < d) {
                    d = v;
                    kb = k;
                }
            } else if (v < disnn[k - r0]) {
                disnn[k - r0] = v;
                nn[k - r0] = I2;
            }
        }
        block_argmin(d, kb, red_d, red_i);
        if (tid == 0) {
            nnc = Cand{d, kb, 0};
            n_list = 0;
        }
        __syncthreads();

        // 3. rescan the rows of this slice whose NN was I2 or J2
        for (int r = r0 + tid; r < r1; r += nt)
            if (r < n - 1 && alive[r] && r != I2 && (nn[r - r0] == I2 || nn[r - r0] == J2))
                list[atomicAdd(&n_list, 1)] = r;
        __syncthreads();
        for (int e = 0; e < n_list; e++) {          // the whole CTA on each row, several loads in flight
            const int r = list[e];
            const double* row = D + (int64_t)r * n;
            double dm = HC_INF;
            int jm = NO_ROW;
            for (int j0 = r + 1 + tid; j0 < n; j0 += 4 * nt) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int j = j0 + u * nt;
                    v[u] = j < n && alive[j] ? __ldcg(row + j) : HC_INF;
                }
#pragma unroll
                for (int u = 0; u < 4; u++)      // ascending j: the lowest index wins ties
                    if (v[u] < dm) {
                        dm = v[u];
                        jm = j0 + u * nt;
                    }
            }
            block_argmin(dm, jm, red_d, red_i);
            if (tid == 0) {
                disnn[r - r0] = dm;
                nn[r - r0] = jm == NO_ROW ? -1 : jm;
            }
        }
        cluster.sync();

        // 4. the new NN of I2, from every CTA's candidate
        if (I2 >= r0 && I2 < r1 && tid == 0) {
            Cand best{HC_INF, NO_ROW, 0};
            for (int q = 0; q < C; q++) {
                const Cand c = *cluster.map_shared_rank(&nnc, q);
                if (c.d < HC_INF && before(c.d, c.i, best.d, best.i)) best = c;
            }
            disnn[I2 - r0] = best.d;
            nn[I2 - r0] = best.i == NO_ROW ? -1 : best.i;
        }
        __syncthreads();
    }
    cluster.sync();     // no CTA leaves while another may still read its shared memory
}

unsigned blocks_of(int64_t n) { return (unsigned)((n + TPB - 1) / TPB); }

// merge and order from IA / IB (0-based rows, IA < IB), in O(n): HCASS2's result
void hcass2(int n, const std::vector<int>& ia, const std::vector<int>& ib, std::vector<int32_t>& merge,
            std::vector<int32_t>& order) {
    const int m = n - 1;
    std::vector<int32_t> last((size_t)n, 0);     // the last step (1-based) that merged into a row
    merge.assign((size_t)2 * m, 0);
    for (int s = 0; s < m; s++) {
        int32_t a = last[ia[s]] ? last[ia[s]] : -(ia[s] + 1);
        int32_t b = last[ib[s]] ? last[ib[s]] : -(ib[s] + 1);
        if (a > 0 && b < 0) std::swap(a, b);                  // a singleton first
        if (a > 0 && b > 0 && a > b) std::swap(a, b);         // two clusters ascending
        merge[s] = a;
        merge[(size_t)m + s] = b;
        last[ia[s]] = s + 1;
    }
    order.clear();
    std::vector<int32_t> stack{m};
    while (!stack.empty()) {
        const int32_t v = stack.back();
        stack.pop_back();
        if (v < 0) {
            order.push_back(-v);
            continue;
        }
        stack.push_back(merge[(size_t)m + v - 1]);            // right child after the left one
        stack.push_back(merge[v - 1]);
    }
}

}  // namespace
}  // namespace rcp

using namespace rcp;

extern "C" int rcp_hclust(const double* x, int64_t n, int64_t p, int64_t ld, int method, int mem, int32_t* merge,
                          double* height, int32_t* order) {
    RCP_TRY(require_ready());
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "hclust: bad mem kind");
    if (n < 2) return fail(RCP_ERR_ARG, "must have n >= 2 objects to cluster");
    if (n > HC_MAX_N) return fail(RCP_ERR_ARG, "size cannot be NA nor exceed 65536");
    if (p < 1 || ld < n) return fail(RCP_ERR_ARG, "hclust: bad shape or leading dimension");
    if (x == nullptr || merge == nullptr || height == nullptr || order == nullptr)
        return fail(RCP_ERR_ARG, "hclust: NULL pointer");
    if (method != RCP_HCLUST_COMPLETE)
        return fail(RCP_ERR_UNSUPPORTED, "hclust: only method = \"complete\" is implemented (got method %d)", method);
    const int N = (int)n;
    DevIn<double> dx;
    RCP_TRY(dx.init(x, (size_t)(p - 1) * (size_t)ld + (size_t)n, mem));

    Arena ar;
    RCP_TRY(ar.reserve(Arena::pad(8) + 2 * Arena::pad((size_t)N * 8) + 3 * Arena::pad((size_t)N * 4)));
    int* flags = ar.take<int>(2);               // [0] non-finite x, [1] a distance >= INF
    double* disnn = ar.take<double>(N);
    double* crit = ar.take<double>(N);
    int* nn = ar.take<int>(N);
    int* d_ia = ar.take<int>(N);
    int* d_ib = ar.take<int>(N);
    int h_flags[2] = {0, 0};
    RCP_CUDA(cudaMemsetAsync(flags, 0, 8, g_ctx.stream));
    hc_finite_kernel<<<std::min(4096u, blocks_of(n * p)), TPB, 0, g_ctx.stream>>>(dx.ptr, n, p, ld, flags);
    RCP_LAUNCHED();
    RCP_CUDA(cudaMemcpyAsync(h_flags, flags, 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    if (h_flags[0]) return fail(RCP_ERR_DATA, "NA/NaN/Inf in foreign function call (arg 1)");

    // the cluster: up to 16 CTAs where the device allows that non-portable size, else up to 8
    static int max_cluster = 0;
    if (max_cluster == 0) {
        RCP_CUDA(cudaFuncSetAttribute(hc_merge_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        max_cluster = 8;
        const size_t smem16 = (size_t)HC_MAX_N + (size_t)(HC_MAX_N / 16) * 16;
        RCP_CUDA(cudaFuncSetAttribute(hc_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem16));
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 16;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3(16);
        cfg.blockDim = dim3(MERGE_THREADS);
        cfg.dynamicSmemBytes = smem16;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int active = 0;
        if (cudaOccupancyMaxActiveClusters(&active, hc_merge_kernel, &cfg) == cudaSuccess && active >= 1)
            max_cluster = 16;
        cudaGetLastError();
    }
    int C = 1;                          // a power of two, about 2 048 rows per CTA
    while (C < max_cluster && (int64_t)C * 2048 < n) C *= 2;
    const int S = (N + C - 1) / C;
    const size_t smem = (size_t)((N + 15) & ~15) + (size_t)S * 16;
    RCP_CUDA(cudaFuncSetAttribute(hc_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    // the full symmetric matrix: every row the merge loop reads is contiguous
    const size_t dbytes = (size_t)n * (size_t)n * 8;
    double* D = nullptr;
    if (device_alloc((void**)&D, dbytes) != RCP_OK) {
        const std::string why = rcp_last_error();
        return fail(RCP_ERR_CUDA, "hclust: the %lld x %lld distance matrix needs %zu bytes of device memory (%s)",
                    (long long)n, (long long)n, dbytes, why.c_str());
    }
    struct FreeD {
        double*& p;
        ~FreeD() { dfree(p); }
    } free_d{D};

    const int64_t T = (n + DT - 1) / DT;
    hc_dist_kernel<<<(unsigned)(T * (T + 1) / 2), TPB, 0, g_ctx.stream>>>(dx.ptr, N, p, ld, D, flags + 1);
    RCP_LAUNCHED();
    RCP_CUDA(cudaMemcpyAsync(h_flags + 1, flags + 1, 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    hc_nn_kernel<<<blocks_of(n * 32), TPB, 0, g_ctx.stream>>>(D, N, disnn, nn);
    RCP_LAUNCHED();
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    if (h_flags[1]) return fail(RCP_ERR_DATA, "hclust: a distance reaches 1e300, hclust's INF");

    {
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)C;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3((unsigned)C);
        cfg.blockDim = dim3(MERGE_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = g_ctx.stream;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        RCP_CUDA(cudaLaunchKernelEx(&cfg, hc_merge_kernel, D, N, S, (const double*)disnn, (const int*)nn, d_ia, d_ib,
                                    crit));
        RCP_LAUNCHED();
    }
    std::vector<int> h_ia((size_t)N - 1), h_ib((size_t)N - 1);
    std::vector<double> h_crit((size_t)N - 1);
    RCP_CUDA(cudaMemcpyAsync(h_ia.data(), d_ia, (size_t)(N - 1) * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(h_ib.data(), d_ib, (size_t)(N - 1) * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(h_crit.data(), crit, (size_t)(N - 1) * 8, cudaMemcpyDeviceToHost, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    dfree(D);

    std::vector<int32_t> h_merge, h_order;
    hcass2(N, h_ia, h_ib, h_merge, h_order);
    const cudaMemcpyKind h2o = mem == RCP_MEM_HOST ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice;
    RCP_CUDA(cudaMemcpyAsync(merge, h_merge.data(), h_merge.size() * 4, h2o, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(height, h_crit.data(), h_crit.size() * 8, h2o, g_ctx.stream));
    RCP_CUDA(cudaMemcpyAsync(order, h_order.data(), h_order.size() * 4, h2o, g_ctx.stream));
    RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return RCP_OK;
}
