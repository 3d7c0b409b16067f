// kmeans(x, centers = k, iter.max, nstart, algorithm) as stats::kmeans runs it for kmeansDesign
// (/root/reference/R/util.R:140-197, recoup.R:602), on the device.
//
// Parity with R's own arithmetic is the goal, so every distance and every centre is formed with
// the floating-point operations of R's kmeans.c / kmns.f in their order: d(i, l) sums
// (x[i,j] - c[l,j])^2 over j in column order, centres sum their members in point order, and
// nothing is contracted into an FMA (explicit __d*_rn intrinsics; the file is also built with
// -fmad=false).  Ties between distances are common in profile matrices (zero rows, repeated bin
// means), and a centre one ulp off decides them differently.
//
//   * all nstart starts run at once, one grid dimension (or one CTA) per start;
//   * Lloyd / Forgy: a parallel assignment kernel over (start, point) and the ordered centre sums
//     (one thread per (start, column) streaming the column), iterated until no point changes;
//   * MacQueen and Hartigan-Wong move one point at a time.  One CTA per start walks the points in
//     chunks: the CTA computes the chunk's distances in parallel, one thread takes the algorithm's
//     decisions from them in point order, and after a transfer L1 -> L2 the CTA rebuilds the two
//     centres elementwise and recomputes the remaining points' distances to L1 and L2.  Every
//     distance is therefore the one R's serial loop computes at that moment; R's early exits
//     (IF (DC .GE. RR) GOTO ...) decide like full sums, since a sum of squares never decreases
//     under rounding.
//
// The random draws (set.seed, sample.int, unique(x)) follow kmeans' own sequence on the host, with
// the library's Mersenne-Twister (r_rng.cuh); unique(x) itself is a device pass (row hashes, a
// radix sort, exact comparison of rows that share a hash, compaction in first-occurrence order).
#include <cmath>
#include <memory>
#include <vector>

#include "r_rng.cuh"
#include "rcp_internal.cuh"

namespace rcp {
namespace {

constexpr int TPB = 256;
constexpr int KM_MAX_K = 256;          // clusters per call (shared-memory accumulators)
constexpr int CEN_THREADS = 64;        // columns per CTA of the centre kernel
constexpr int WALK_THREADS = 512;
constexpr size_t WALK_SMEM_MAX = 200 * 1024;
constexpr double BIG = 1.0e30;

// d(i, l) with R's operations: tmp = x - c; dd += tmp * tmp, columns in order.  c points at
// centre l of a column-major k x p centre matrix.
__device__ __forceinline__ double sqdist(const double* __restrict__ xi, int64_t ld, const double* c, int k,
                                         int64_t p) {
    double d = 0.0;
    for (int64_t j = 0; j < p; j++) {
        const double t = __dsub_rn(xi[j * ld], c[j * k]);
        d = __dadd_rn(d, __dmul_rn(t, t));
    }
    return d;
}

// the same for G consecutive centres l0 .. l0+G-1 at once (one read of the row)
template <int G>
__device__ __forceinline__ void sqdist_group(const double* __restrict__ xi, int64_t ld, const double* c, int k,
                                             int64_t p, int l0, double* acc) {
    const int nu = min(G, k - l0);
#pragma unroll
    for (int u = 0; u < G; u++) acc[u] = 0.0;
    for (int64_t j = 0; j < p; j++) {
        const double xv = xi[j * ld];
        const double* cj = c + j * k + l0;
#pragma unroll
        for (int u = 0; u < G; u++)
            if (u < nu) {
                const double t = __dsub_rn(xv, cj[u]);
                acc[u] = __dadd_rn(acc[u], __dmul_rn(t, t));
            }
    }
}

__global__ void __launch_bounds__(TPB)
km_finite_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld, int* __restrict__ bad) {
    const int64_t n = m * p;
    for (int64_t t = (int64_t)blockIdx.x * TPB + threadIdx.x; t < n; t += (int64_t)gridDim.x * TPB) {
        const int64_t j = t / m, i = t - j * m;
        if (!isfinite(x[i + j * ld])) {
            *bad = 1;
            return;
        }
    }
}

// ---- unique(x) ------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB)
km_row_hash_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld,
                   unsigned long long* __restrict__ keys, int32_t* __restrict__ rows) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= m) return;
    unsigned long long h = 0x9e3779b97f4a7c15ull;
    for (int64_t j = 0; j < p; j++) {
        // -0.0 + 0.0 = +0.0: the two zeros hash alike, as they compare equal
        const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(x[i + j * ld], 0.0));
        h = (h ^ b) * 0xbf58476d1ce4e5b9ull;
        h ^= h >> 31;
    }
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    keys[i] = h;
    rows[i] = (int32_t)i;
}

// first[row] = 1 iff no row of smaller index equals it.  The sort is stable, so within a run of
// equal hashes the rows are in index order; a duplicate usually meets its equal right before it.
__global__ void __launch_bounds__(TPB)
km_first_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld,
                const unsigned long long* __restrict__ keys, const int32_t* __restrict__ rows,
                uint32_t* __restrict__ first) {
    const int64_t t = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (t >= m) return;
    const int64_t a = rows[t];
    uint32_t is_first = 1;
    for (int64_t u = t - 1; u >= 0 && keys[u] == keys[t] && is_first; u--) {
        const int64_t b = rows[u];
        bool eq = true;
        for (int64_t j = 0; j < p && eq; j++) eq = x[a + j * ld] == x[b + j * ld];
        if (eq) is_first = 0;
    }
    first[a] = is_first;
}

__global__ void __launch_bounds__(TPB)
km_compact_kernel(int64_t m, const uint32_t* __restrict__ first, const uint32_t* __restrict__ at,
                  int32_t* __restrict__ uidx) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i < m && first[i]) uidx[at[i]] = (int32_t)i;
}

// initial centres of every start: cen[s][j*k + l] = x[row(s, l), j]; pos are 1-based positions
// into the rows (uidx == nullptr) or into the distinct rows
__global__ void __launch_bounds__(TPB)
km_gather_kernel(const double* __restrict__ x, int64_t p, int64_t ld, int k, const int32_t* __restrict__ pos,
                 const int32_t* __restrict__ uidx, double* __restrict__ cen) {
    const int s = blockIdx.y;
    const int64_t t = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (t >= (int64_t)k * p) return;
    const int64_t j = t / k;
    const int l = (int)(t - j * k);
    const int32_t q = pos[s * k + l] - 1;
    const int64_t row = uidx ? uidx[q] : q;
    cen[(int64_t)s * k * p + t] = x[row + j * ld];
}

// ---- assignment ---------------------------------------------------------------------------
// HW == false: cl = the first centre with the strictly smallest distance (kmeans_Lloyd /
//   kmeans_MacQueen); a change raises upd[s * upd_stride].  Starts with done[s] set are skipped.
// HW == true: the IC1 / IC2 set-up of kmns (k >= 2).
template <bool HW>
__global__ void __launch_bounds__(TPB)
km_assign_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld, int k,
                 const double* __restrict__ cen, int32_t* __restrict__ cl, int32_t* __restrict__ ic2,
                 const int* __restrict__ done, int* __restrict__ upd, int upd_stride) {
    const int s = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= m || (done && done[s])) return;
    const double* c = cen + (int64_t)s * k * p;
    const double* xi = x + i;
    double acc[8];
    if (!HW) {
        double best = INFINITY;
        int inew = 0;
        for (int l0 = 0; l0 < k; l0 += 8) {
            sqdist_group<8>(xi, ld, c, k, p, l0, acc);
            for (int u = 0; u < 8 && l0 + u < k; u++)
                if (acc[u] < best) {
                    best = acc[u];
                    inew = l0 + u;
                }
        }
        int32_t* me = cl + (int64_t)s * m + i;
        if (*me != inew) {
            *me = inew;
            if (upd) upd[s * upd_stride] = 1;
        }
        return;
    }
    int c1 = 0, c2 = 1;
    double dt1 = 0.0, dt2 = 0.0;
    for (int l0 = 0; l0 < k; l0 += 8) {
        sqdist_group<8>(xi, ld, c, k, p, l0, acc);
        for (int u = 0; u < 8 && l0 + u < k; u++) {
            const int l = l0 + u;
            const double db = acc[u];
            if (l == 0) {
                dt1 = db;
            } else if (l == 1) {
                dt2 = db;
                if (dt1 > dt2) {
                    c1 = 1;
                    c2 = 0;
                    const double t = dt1;
                    dt1 = dt2;
                    dt2 = t;
                }
            } else if (db < dt2) {
                if (db < dt1) {
                    dt2 = dt1;
                    c2 = c1;
                    dt1 = db;
                    c1 = l;
                } else {
                    dt2 = db;
                    c2 = l;
                }
            }
        }
    }
    cl[(int64_t)s * m + i] = c1;
    ic2[(int64_t)s * m + i] = c2;
}

// ---- centres as means -------------------------------------------------------------------
// One thread per (start, column): the members of every cluster are added in point order, then
// divided by the count (0 / 0 = NaN for an empty cluster, as in R).  nc (optional) receives the
// counts.  Lloyd: a start without a change in this iteration is finished (iter = it + 1).
__global__ void __launch_bounds__(CEN_THREADS)
km_centres_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld, int k,
                  const int32_t* __restrict__ cl, double* __restrict__ cen, int32_t* __restrict__ nc,
                  int* __restrict__ done, const int* __restrict__ upd, int upd_stride,
                  int* __restrict__ iter_out, int it) {
    extern __shared__ double sh[];
    const int s = blockIdx.y;
    if (done && done[s]) return;
    if (upd && !upd[s * upd_stride]) {
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            done[s] = 1;
            iter_out[s] = it + 1;
        }
        return;
    }
    const int t = threadIdx.x;
    const int64_t j = (int64_t)blockIdx.x * CEN_THREADS + t;
    if (j >= p) return;
    double* acc = sh + t;
    int* cnt = reinterpret_cast<int*>(sh + (size_t)k * CEN_THREADS) + t;
    for (int l = 0; l < k; l++) {
        acc[l * CEN_THREADS] = 0.0;
        cnt[l * CEN_THREADS] = 0;
    }
    const int32_t* c = cl + (int64_t)s * m;
    const double* xc = x + j * ld;
    int64_t i = 0;
    for (; i + 4 <= m; i += 4) {          // loads first, then the adds in point order
        const int l0 = c[i], l1 = c[i + 1], l2 = c[i + 2], l3 = c[i + 3];
        const double v0 = xc[i], v1 = xc[i + 1], v2 = xc[i + 2], v3 = xc[i + 3];
        acc[l0 * CEN_THREADS] = __dadd_rn(acc[l0 * CEN_THREADS], v0);
        cnt[l0 * CEN_THREADS]++;
        acc[l1 * CEN_THREADS] = __dadd_rn(acc[l1 * CEN_THREADS], v1);
        cnt[l1 * CEN_THREADS]++;
        acc[l2 * CEN_THREADS] = __dadd_rn(acc[l2 * CEN_THREADS], v2);
        cnt[l2 * CEN_THREADS]++;
        acc[l3 * CEN_THREADS] = __dadd_rn(acc[l3 * CEN_THREADS], v3);
        cnt[l3 * CEN_THREADS]++;
    }
    for (; i < m; i++) {
        const int l = c[i];
        acc[l * CEN_THREADS] = __dadd_rn(acc[l * CEN_THREADS], xc[i]);
        cnt[l * CEN_THREADS]++;
    }
    double* out = cen + (int64_t)s * k * p + j * k;
    for (int l = 0; l < k; l++) {
        out[l] = __ddiv_rn(acc[l * CEN_THREADS], (double)cnt[l * CEN_THREADS]);
        if (nc && j == 0) nc[s * k + l] = cnt[l * CEN_THREADS];
    }
}

// ---- the serial algorithms: one CTA per start ---------------------------------------------
struct WalkArgs {
    const double* x;
    int64_t m, p, ld;
    int k, iter_max, chunk;
    long long imaxqtr;
    bool cen_smem;
    double* cen;     // S x (k x p)
    int32_t* cl;     // S x m   (IC1)
    int32_t* ic2;    // S x m   (Hartigan-Wong)
    double* D;       // S x m   (Hartigan-Wong)
    int32_t* nc;     // S x k
    int* iter_out;   // S
    int* ifault;     // S
};

struct WalkCtl {
    int tr;          // chunk position of the transfer the walker stopped at, -1 = none
    int l1, l2;
    int ret;         // 1: the stage returned (HW: INDX == M / ICOUN == M), 2: quick-transfer limit
    int updated;     // MacQueen: a point moved in this pass
    long long istep; // QTRAN: thread 0's step count
    double al1, alw, al2, alt;
};

struct WalkSmem {
    double* cen;     // centres (shared or global)
    double* dist;    // chunk x k (OPTRA, MacQueen); QTRAN uses columns 0 and 1
    double* cD;
    int32_t *c1, *c2;
    double *an1, *an2;
    int32_t *ncs, *itran;
    long long *ncp, *live;
    WalkCtl* ctl;
};

__host__ __device__ inline size_t walk_smem_bytes(int k, int64_t p, int chunk, bool cen_smem) {
    size_t b = (size_t)chunk * k * 8 + (size_t)chunk * (8 + 4 + 4) + (size_t)k * (8 + 8 + 4 + 4 + 8 + 8) +
               sizeof(WalkCtl) + 64;
    if (cen_smem) b += (size_t)k * p * 8;
    return b;
}

__device__ __forceinline__ WalkSmem walk_layout(char* base, const WalkArgs& a, double* gcen) {
    WalkSmem w;
    const int k = a.k, C = a.chunk;
    char* q = base;
    auto take = [&](size_t bytes) {
        char* r = q;
        q += (bytes + 7) & ~(size_t)7;
        return r;
    };
    w.ctl = reinterpret_cast<WalkCtl*>(take(sizeof(WalkCtl)));
    w.dist = reinterpret_cast<double*>(take((size_t)C * k * 8));
    w.cD = reinterpret_cast<double*>(take((size_t)C * 8));
    w.an1 = reinterpret_cast<double*>(take((size_t)k * 8));
    w.an2 = reinterpret_cast<double*>(take((size_t)k * 8));
    w.ncp = reinterpret_cast<long long*>(take((size_t)k * 8));
    w.live = reinterpret_cast<long long*>(take((size_t)k * 8));
    w.c1 = reinterpret_cast<int32_t*>(take((size_t)C * 4));
    w.c2 = reinterpret_cast<int32_t*>(take((size_t)C * 4));
    w.ncs = reinterpret_cast<int32_t*>(take((size_t)k * 4));
    w.itran = reinterpret_cast<int32_t*>(take((size_t)k * 4));
    w.cen = a.cen_smem ? reinterpret_cast<double*>(take((size_t)k * a.p * 8)) : gcen;
    return w;
}

// centres L1 (a point left it) and L2 (it joined) after a transfer of point i, elementwise
template <bool HW>
__device__ __forceinline__ void walk_move(const WalkArgs& a, const WalkSmem& w, int64_t i) {
    const WalkCtl c = *w.ctl;
    const int k = a.k;
    for (int64_t j = threadIdx.x; j < a.p; j += WALK_THREADS) {
        const double xv = a.x[i + j * a.ld];
        double* p1 = w.cen + j * k + c.l1;
        double* p2 = w.cen + j * k + c.l2;
        if (HW) {       // C(L1,J) = (C(L1,J) * AL1 - A(I,J)) / ALW;  C(L2,J) = (C(L2,J) * AL2 + A(I,J)) / ALT
            *p1 = __ddiv_rn(__dsub_rn(__dmul_rn(*p1, c.al1), xv), c.alw);
            *p2 = __ddiv_rn(__dadd_rn(__dmul_rn(*p2, c.al2), xv), c.alt);
        } else {        // cen[old] += (cen[old] - x) / nc[old];  cen[new] += (x - cen[new]) / nc[new]
            *p1 = __dadd_rn(*p1, __ddiv_rn(__dsub_rn(*p1, xv), c.al1));
            *p2 = __dadd_rn(*p2, __ddiv_rn(__dsub_rn(xv, *p2), c.al2));
        }
    }
}

// chunk loads / stores between the start's global arrays and shared memory
__device__ __forceinline__ void walk_load(const WalkArgs& a, const WalkSmem& w, int s, int64_t c0, int n, bool hw) {
    for (int t = threadIdx.x; t < n; t += WALK_THREADS) {
        w.c1[t] = a.cl[(int64_t)s * a.m + c0 + t];
        if (hw) {
            w.c2[t] = a.ic2[(int64_t)s * a.m + c0 + t];
            w.cD[t] = a.D[(int64_t)s * a.m + c0 + t];
        }
    }
}
__device__ __forceinline__ void walk_store(const WalkArgs& a, const WalkSmem& w, int s, int64_t c0, int n, bool hw) {
    for (int t = threadIdx.x; t < n; t += WALK_THREADS) {
        a.cl[(int64_t)s * a.m + c0 + t] = w.c1[t];
        if (hw) {
            a.ic2[(int64_t)s * a.m + c0 + t] = w.c2[t];
            a.D[(int64_t)s * a.m + c0 + t] = w.cD[t];
        }
    }
}

// distances of chunk points [from, n) to every centre (l_a < 0) or to centres l_a and l_b
__device__ __forceinline__ void walk_dist(const WalkArgs& a, const WalkSmem& w, int64_t c0, int from, int n,
                                          int l_a, int l_b) {
    const int k = a.k;
    const int rem = n - from;
    if (rem <= 0) return;
    const int nl = l_a < 0 ? k : 2;
    for (int task = threadIdx.x; task < rem * nl; task += WALK_THREADS) {
        const int t = from + task % rem;
        const int u = task / rem;
        const int l = l_a < 0 ? u : (u == 0 ? l_a : l_b);
        w.dist[t * k + l] = sqdist(a.x + c0 + t, a.ld, w.cen + l, k, a.p);
    }
}

// kmeans_MacQueen after its set-up (nearest-centre assignment and means, done by the kernels above)
__device__ void walk_macqueen(const WalkArgs& a, const WalkSmem& w, int s) {
    const int k = a.k;
    int inew = 0;                        // carried from point to point, as in kmeans.c
    int iter = 0;
    for (; iter < a.iter_max; iter++) {
        if (threadIdx.x == 0) w.ctl->updated = 0;
        for (int64_t c0 = 0; c0 < a.m; c0 += a.chunk) {
            const int n = (int)min((int64_t)a.chunk, a.m - c0);
            walk_load(a, w, s, c0, n, false);
            walk_dist(a, w, c0, 0, n, -1, -1);
            __syncthreads();
            int q = 0;
            for (;;) {
                if (threadIdx.x == 0) {
                    WalkCtl* c = w.ctl;
                    c->tr = -1;
                    for (int t = q; t < n; t++) {
                        double best = INFINITY;
                        for (int l = 0; l < k; l++) {
                            const double dd = w.dist[t * k + l];
                            if (dd < best) {
                                best = dd;
                                inew = l;
                            }
                        }
                        const int iold = w.c1[t];
                        if (iold != inew) {
                            c->updated = 1;
                            w.c1[t] = inew;
                            w.ncs[iold]--;
                            w.ncs[inew]++;
                            c->tr = t;
                            c->l1 = iold;
                            c->l2 = inew;
                            c->al1 = (double)w.ncs[iold];
                            c->al2 = (double)w.ncs[inew];
                            break;
                        }
                    }
                }
                __syncthreads();
                const int tr = w.ctl->tr;
                if (tr < 0) break;
                const int l1 = w.ctl->l1, l2 = w.ctl->l2;
                walk_move<false>(a, w, c0 + tr);
                __syncthreads();
                walk_dist(a, w, c0, tr + 1, n, l1, l2);
                q = tr + 1;
                __syncthreads();
            }
            walk_store(a, w, s, c0, n, false);
            __syncthreads();
        }
        const int updated = w.ctl->updated;
        __syncthreads();
        if (!updated) break;
    }
    if (threadIdx.x == 0) a.iter_out[s] = iter + 1;
}

// the transfer of chunk point t from L1 to L2, common to OPTRA and QTRAN (thread 0): counts, AN1 /
// AN2, IC1 / IC2, and the factors walk_move needs
__device__ __forceinline__ void hw_transfer(const WalkSmem& w, WalkCtl* ctl, int t, int L1, int L2) {
    const double al1 = (double)w.ncs[L1], alw = __dsub_rn(al1, 1.0);
    const double al2 = (double)w.ncs[L2], alt = __dadd_rn(al2, 1.0);
    w.ncs[L1]--;
    w.ncs[L2]++;
    w.an2[L1] = __ddiv_rn(alw, al1);
    w.an1[L1] = alw > 1.0 ? __ddiv_rn(alw, __dsub_rn(alw, 1.0)) : BIG;
    w.an1[L2] = __ddiv_rn(alt, al2);
    w.an2[L2] = __ddiv_rn(alt, __dadd_rn(alt, 1.0));
    w.c1[t] = L2;
    w.c2[t] = L1;
    ctl->tr = t;
    ctl->l1 = L1;
    ctl->l2 = L2;
    ctl->al1 = al1;
    ctl->alw = alw;
    ctl->al2 = al2;
    ctl->alt = alt;
}

// QTRAN's distances of chunk points [from, n): dist[t*k] = d(i, IC1) when the step of point t will
// recompute D(I) (ISTEP <= NCP(L1)), dist[t*k + 1] = d(i, IC2) when it will test a transfer
// (ISTEP < NCP(L1) or ISTEP < NCP(L2)).  istep_base = the step count before point `from`.  With
// la >= 0 only the points that reference cluster la or lb are recomputed (the others' centres and
// conditions did not change).
__device__ __forceinline__ void qtran_prepare(const WalkArgs& a, const WalkSmem& w, int64_t c0, int n, int from,
                                              long long istep_base, int la, int lb) {
    const int k = a.k;
    const int rem = n - from;
    for (int task = threadIdx.x; task < 2 * rem; task += WALK_THREADS) {
        const int t = from + task % rem;
        const int which = task / rem;
        const int L1 = w.c1[t], L2 = w.c2[t];
        if (la >= 0 && L1 != la && L1 != lb && L2 != la && L2 != lb) continue;
        if (w.ncs[L1] == 1) continue;
        const long long st = istep_base + (t - from) + 1;
        const bool need = which == 0 ? st <= w.ncp[L1] : (st < w.ncp[L1] || st < w.ncp[L2]);
        if (need) w.dist[t * k + which] = sqdist(a.x + c0 + t, a.ld, w.cen + (which == 0 ? L1 : L2), k, a.p);
    }
}

// AS 136 (kmns) main loop after its set-up (IC1 / IC2 and the means, done by the kernels above)
__device__ void walk_hartigan_wong(const WalkArgs& a, const WalkSmem& w, int s) {
    const int k = a.k;
    const int64_t m = a.m;
    WalkCtl* ctl = w.ctl;
    if (threadIdx.x == 0) {
        int empty = 0;
        for (int l = 0; l < k; l++) empty |= w.ncs[l] == 0;
        ctl->ret = empty;
        if (empty) a.ifault[s] = 1;
        for (int l = 0; l < k; l++) {
            const double aa = (double)w.ncs[l];
            w.an2[l] = __ddiv_rn(aa, __dadd_rn(aa, 1.0));
            w.an1[l] = aa > 1.0 ? __ddiv_rn(aa, __dsub_rn(aa, 1.0)) : BIG;
            w.itran[l] = 1;
            w.ncp[l] = -1;
        }
    }
    __syncthreads();
    if (ctl->ret) return;
    long long indx = 0;                  // thread 0's walker state
    int result_iter = a.iter_max + 1, result_fault = 2;
    for (int ij = 1; ij <= a.iter_max; ij++) {
        // ---- OPTRA: the optimal-transfer stage, one pass through the data
        if (threadIdx.x == 0)
            for (int l = 0; l < k; l++)
                if (w.itran[l] == 1) w.live[l] = m + 1;
        int returned = 0;
        for (int64_t c0 = 0; c0 < m && !returned; c0 += a.chunk) {
            const int n = (int)min((int64_t)a.chunk, m - c0);
            walk_load(a, w, s, c0, n, true);
            walk_dist(a, w, c0, 0, n, -1, -1);
            __syncthreads();
            int q = 0;
            for (;;) {
                if (threadIdx.x == 0) {
                    ctl->tr = -1;
                    ctl->ret = 0;
                    for (int t = q; t < n; t++) {
                        const long long i1 = c0 + t + 1;
                        indx++;
                        const int L1 = w.c1[t];
                        if (w.ncs[L1] != 1) {
                            const double* dr = w.dist + t * k;
                            if (w.ncp[L1] != 0) w.cD[t] = __dmul_rn(dr[L1], w.an1[L1]);
                            int L2 = w.c2[t];
                            const int LL = L2;
                            double r2 = __dmul_rn(dr[L2], w.an2[L2]);
                            for (int l = 0; l < k; l++) {
                                if ((i1 >= w.live[L1] && i1 >= w.live[l]) || l == L1 || l == LL) continue;
                                const double rr = __ddiv_rn(r2, w.an2[l]);
                                if (dr[l] < rr) {
                                    r2 = __dmul_rn(dr[l], w.an2[l]);
                                    L2 = l;
                                }
                            }
                            if (r2 >= w.cD[t]) {
                                w.c2[t] = L2;
                            } else {
                                indx = 0;
                                w.live[L1] = m + i1;
                                w.live[L2] = m + i1;
                                w.ncp[L1] = i1;
                                w.ncp[L2] = i1;
                                hw_transfer(w, ctl, t, L1, L2);
                                break;
                            }
                        }
                        if (indx == m) {
                            ctl->ret = 1;
                            break;
                        }
                    }
                }
                __syncthreads();
                const int tr = ctl->tr;
                if (tr < 0) {
                    returned = ctl->ret;
                    break;
                }
                const int l1 = ctl->l1, l2 = ctl->l2;
                walk_move<true>(a, w, c0 + tr);
                __syncthreads();
                walk_dist(a, w, c0, tr + 1, n, l1, l2);
                q = tr + 1;
                __syncthreads();
            }
            walk_store(a, w, s, c0, n, true);
            __syncthreads();
        }
        if (threadIdx.x == 0 && !returned)
            for (int l = 0; l < k; l++) {
                w.itran[l] = 0;
                w.live[l] -= m;
            }
        if (returned) {                  // INDX == M: no transfer in the last M steps
            result_iter = ij;
            result_fault = 0;
            break;
        }
        // ---- QTRAN: the quick-transfer stage.  dist[t*k + 0] = d(i, IC1), [t*k + 1] = d(i, IC2),
        // computed for the points whose step will need them
        long long icoun = 0, istep = 0;
        int qret = 0;
        for (int64_t c0 = 0; !qret; c0 = (c0 + a.chunk >= m) ? 0 : c0 + a.chunk) {   // GO TO 10: wrap
            const int n = (int)min((int64_t)a.chunk, m - c0);
            walk_load(a, w, s, c0, n, true);
            if (threadIdx.x == 0) ctl->istep = istep;
            __syncthreads();
            qtran_prepare(a, w, c0, n, 0, ctl->istep, -1, -1);
            __syncthreads();
            int q = 0;
            for (;;) {
                if (threadIdx.x == 0) {
                    ctl->tr = -1;
                    ctl->ret = 0;
                    for (int t = q; t < n; t++) {
                        icoun++;
                        istep++;
                        if (istep >= a.imaxqtr) {
                            ctl->ret = 2;
                            break;
                        }
                        const int L1 = w.c1[t], L2 = w.c2[t];
                        if (w.ncs[L1] != 1) {
                            if (istep <= w.ncp[L1]) w.cD[t] = __dmul_rn(w.dist[t * k], w.an1[L1]);
                            if (istep < w.ncp[L1] || istep < w.ncp[L2]) {
                                const double r2 = __ddiv_rn(w.cD[t], w.an2[L2]);
                                if (w.dist[t * k + 1] < r2) {
                                    icoun = 0;
                                    indx = 0;
                                    w.itran[L1] = 1;
                                    w.itran[L2] = 1;
                                    w.ncp[L1] = istep + m;
                                    w.ncp[L2] = istep + m;
                                    hw_transfer(w, ctl, t, L1, L2);
                                    break;
                                }
                            }
                        }
                        if (icoun == m) {
                            ctl->ret = 1;
                            break;
                        }
                    }
                    ctl->istep = istep;
                }
                __syncthreads();
                const int tr = ctl->tr;
                if (tr < 0) {
                    qret = ctl->ret;
                    break;
                }
                const int l1 = ctl->l1, l2 = ctl->l2;
                const long long ist = ctl->istep;
                walk_move<true>(a, w, c0 + tr);
                __syncthreads();
                qtran_prepare(a, w, c0, n, tr + 1, ist, l1, l2);
                q = tr + 1;
                __syncthreads();
            }
            walk_store(a, w, s, c0, n, true);
            __syncthreads();
        }
        if (qret == 2) {                 // IMAXQTR steps: IFAULT = 4
            result_iter = ij;
            result_fault = 4;
            break;
        }
        if (k == 2) {
            result_iter = ij;
            result_fault = 0;
            break;
        }
        if (threadIdx.x == 0)
            for (int l = 0; l < k; l++) w.ncp[l] = 0;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.iter_out[s] = result_iter;
        a.ifault[s] = result_fault;
    }
}

template <bool HW>
__global__ void __launch_bounds__(WALK_THREADS) km_walk_kernel(WalkArgs a) {
    extern __shared__ __align__(16) char smem[];
    const int s = blockIdx.x;
    double* gcen = a.cen + (int64_t)s * a.k * a.p;
    const WalkSmem w = walk_layout(smem, a, gcen);
    if (a.cen_smem)
        for (int64_t t = threadIdx.x; t < (int64_t)a.k * a.p; t += WALK_THREADS) w.cen[t] = gcen[t];
    for (int l = threadIdx.x; l < a.k; l += WALK_THREADS) w.ncs[l] = a.nc[s * a.k + l];
    __syncthreads();
    if (HW)
        walk_hartigan_wong(a, w, s);
    else
        walk_macqueen(a, w, s);
    __syncthreads();
    if (a.cen_smem)
        for (int64_t t = threadIdx.x; t < (int64_t)a.k * a.p; t += WALK_THREADS) gcen[t] = w.cen[t];
    for (int l = threadIdx.x; l < a.k; l += WALK_THREADS) a.nc[s * a.k + l] = w.ncs[l];
}

// ---- within-cluster sums of squares, sizes, totss ----------------------------------------
__global__ void __launch_bounds__(TPB)
km_err_kernel(const double* __restrict__ x, int64_t m, int64_t p, int64_t ld, int k, const double* __restrict__ cen,
              const int32_t* __restrict__ cl, double* __restrict__ e) {
    const int s = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= m) return;
    const int l = cl[(int64_t)s * m + i];
    e[(int64_t)s * m + i] = sqdist(x + i, ld, cen + (int64_t)s * k * p + l, k, p);
}

__device__ __forceinline__ double block_sum(double v, double* sh) {
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < TPB / 32; w++) t += sh[w];
    return t;
}

// one CTA per (start, cluster): wss = sum of the members' squared distances, nc = members
__global__ void __launch_bounds__(TPB)
km_wss_kernel(int64_t m, int k, const int32_t* __restrict__ cl, const double* __restrict__ e,
              double* __restrict__ wss, int32_t* __restrict__ nc) {
    __shared__ double sh[TPB / 32];
    const int l = blockIdx.x, s = blockIdx.y;
    double v = 0.0, n = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += TPB)
        if (cl[(int64_t)s * m + i] == l) {
            v += e[(int64_t)s * m + i];
            n += 1.0;
        }
    v = block_sum(v, sh);
    n = block_sum(n, sh);
    if (threadIdx.x == 0) {
        wss[s * k + l] = v;
        nc[s * k + l] = (int32_t)n;
    }
}

// totss = sum(scale(x, scale = FALSE)^2): per column, sum of squared deviations from the mean
__global__ void __launch_bounds__(TPB)
km_colss_kernel(const double* __restrict__ x, int64_t m, int64_t ld, double* __restrict__ colss) {
    __shared__ double sh[TPB / 32];
    const double* c = x + (int64_t)blockIdx.x * ld;
    double v = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += TPB) v += c[i];
    const double mean = block_sum(v, sh) / (double)m;
    double q = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += TPB) {
        const double d = c[i] - mean;
        q += d * d;
    }
    q = block_sum(q, sh);
    if (threadIdx.x == 0) colss[blockIdx.x] = q;
}

__global__ void __launch_bounds__(TPB)
km_cluster_out_kernel(int64_t m, const int32_t* __restrict__ cl, int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i < m) out[i] = cl[i] + 1;
}

unsigned blocks_for(int64_t n) { return (unsigned)((n + TPB - 1) / TPB); }

// Distinct rows of x in first-occurrence order -> *uidx (device, mm entries), *mm (host).
int unique_rows(const double* x, int64_t m, int64_t p, int64_t ld, int32_t** uidx, int64_t* mm) {
    unsigned long long* keys = nullptr;
    int32_t* rows = nullptr;
    uint32_t *first = nullptr, *at = nullptr, *total = nullptr;
    RCP_TRY(dalloc(&keys, (size_t)m));
    RCP_TRY(dalloc(&rows, (size_t)m));
    km_row_hash_kernel<<<blocks_for(m), TPB, 0, g_ctx.stream>>>(x, m, p, ld, keys, rows);
    RCP_LAUNCHED();
    int rc = sort_pairs(keys, rows, m, 0, 64);
    if (rc == RCP_OK) rc = dalloc(&first, (size_t)m);
    if (rc == RCP_OK) rc = dalloc(&at, (size_t)m);
    if (rc == RCP_OK) rc = dalloc(&total, 1);
    if (rc == RCP_OK) rc = dalloc(uidx, (size_t)m);
    if (rc == RCP_OK) {
        km_first_kernel<<<blocks_for(m), TPB, 0, g_ctx.stream>>>(x, m, p, ld, keys, rows, first);
        g_ctx.launches++;
        rc = exclusive_scan_u32(first, at, m, total);
    }
    uint32_t h_total = 0;
    if (rc == RCP_OK) {
        km_compact_kernel<<<blocks_for(m), TPB, 0, g_ctx.stream>>>(m, first, at, *uidx);
        g_ctx.launches++;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_total, total, 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "kmeans: unique(x) failed: %s", cudaGetErrorString(e));
    }
    dfree(keys);
    dfree(rows);
    dfree(first);
    dfree(at);
    dfree(total);
    *mm = h_total;
    return rc;
}

// Per-call device state.
struct KmState {
    int64_t m = 0, p = 0, ld = 0;
    int k = 0, S = 0;
    double* cen = nullptr;     // S x k x p
    int32_t* cl = nullptr;     // S x m
    int32_t* ic2 = nullptr;
    double* D = nullptr;
    int32_t* nc = nullptr;     // S x k
    int* iter = nullptr;       // S
    int* ifault = nullptr;     // S
    ~KmState() {
        dfree(cen);
        dfree(cl);
        dfree(ic2);
        dfree(D);
        dfree(nc);
        dfree(iter);
        dfree(ifault);
    }
};

int run_lloyd(const double* x, KmState& st, int iter_max) {
    const int S = st.S, k = st.k;
    int *done = nullptr, *upd = nullptr;
    RCP_TRY(dalloc(&done, (size_t)S));
    RCP_TRY(dalloc(&upd, (size_t)S * iter_max));
    int rc = RCP_OK;
    const size_t smem = (size_t)k * CEN_THREADS * 12;
    cudaError_t e = cudaFuncSetAttribute(km_centres_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaMemsetAsync(done, 0, (size_t)S * 4, g_ctx.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(upd, 0, (size_t)S * iter_max * 4, g_ctx.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(st.cl, 0xff, (size_t)S * st.m * 4, g_ctx.stream);   // cl = -1
    if (e != cudaSuccess) rc = fail(RCP_ERR_CUDA, "kmeans (Lloyd) set-up: %s", cudaGetErrorString(e));
    const dim3 ga(blocks_for(st.m), S), gc((unsigned)((st.p + CEN_THREADS - 1) / CEN_THREADS), S);
    for (int it = 0; it < iter_max && rc == RCP_OK; it++) {
        km_assign_kernel<false><<<ga, TPB, 0, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cen, st.cl, nullptr, done,
                                                              upd + it, iter_max);
        km_centres_kernel<<<gc, CEN_THREADS, smem, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cl, st.cen, nullptr,
                                                                   done, upd + it, iter_max, st.iter, it);
        g_ctx.launches += 2;
        if ((e = cudaGetLastError()) != cudaSuccess)
            rc = fail(RCP_ERR_CUDA, "kmeans (Lloyd) launch: %s", cudaGetErrorString(e));
    }
    dfree(done);
    dfree(upd);
    return rc;
}

int run_walk(const double* x, KmState& st, int iter_max, bool hw) {
    const int S = st.S, k = st.k;
    const size_t csmem = (size_t)k * CEN_THREADS * 12;
    RCP_CUDA(cudaFuncSetAttribute(km_centres_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csmem));
    const dim3 ga(blocks_for(st.m), S), gc((unsigned)((st.p + CEN_THREADS - 1) / CEN_THREADS), S);
    if (hw)
        km_assign_kernel<true><<<ga, TPB, 0, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cen, st.cl, st.ic2, nullptr,
                                                             nullptr, 0);
    else
        km_assign_kernel<false><<<ga, TPB, 0, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cen, st.cl, nullptr,
                                                              nullptr, nullptr, 0);
    RCP_LAUNCHED();
    km_centres_kernel<<<gc, CEN_THREADS, csmem, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cl, st.cen, st.nc,
                                                                nullptr, nullptr, 0, nullptr, 0);
    RCP_LAUNCHED();
    WalkArgs a;
    a.x = x;
    a.m = st.m;
    a.p = st.p;
    a.ld = st.ld;
    a.k = k;
    a.iter_max = iter_max;
    a.chunk = (int)std::min<int64_t>(128, std::max<int64_t>(16, 8192 / k));
    a.imaxqtr = std::min<long long>(0x7fffffffLL, 50LL * st.m);
    a.cen = st.cen;
    a.cl = st.cl;
    a.ic2 = st.ic2;
    a.D = st.D;
    a.nc = st.nc;
    a.iter_out = st.iter;
    a.ifault = st.ifault;
    a.cen_smem = walk_smem_bytes(k, st.p, a.chunk, true) <= WALK_SMEM_MAX;
    const size_t smem = walk_smem_bytes(k, st.p, a.chunk, a.cen_smem);
    if (hw) {
        RCP_CUDA(cudaMemsetAsync(st.D, 0, (size_t)S * st.m * 8, g_ctx.stream));
        RCP_CUDA(cudaFuncSetAttribute(km_walk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        km_walk_kernel<true><<<S, WALK_THREADS, smem, g_ctx.stream>>>(a);
    } else {
        RCP_CUDA(cudaFuncSetAttribute(km_walk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        km_walk_kernel<false><<<S, WALK_THREADS, smem, g_ctx.stream>>>(a);
    }
    RCP_LAUNCHED();
    if (hw) {   // kmns ends by recomputing the centres from scratch, members in point order
        km_centres_kernel<<<gc, CEN_THREADS, csmem, g_ctx.stream>>>(x, st.m, st.p, st.ld, k, st.cl, st.cen, nullptr,
                                                                    nullptr, nullptr, 0, nullptr, 0);
        RCP_LAUNCHED();
    }
    return RCP_OK;
}

bool rows_equal(const double* a, const double* b, int k, int64_t p, int la, int lb) {
    for (int64_t j = 0; j < p; j++)
        if (!(a[j * k + la] == b[j * k + lb])) return false;
    return true;
}

}  // namespace
}  // namespace rcp

using namespace rcp;

extern "C" int rcp_kmeans(const double* x, int64_t m, int64_t p, int64_t ld, int k, int nstart, int iter_max,
                          int algorithm, int seed, int sample_kind, int mem, int32_t* cluster, double* centers,
                          double* withinss, int32_t* size, double* totss, int* iter, int* ifault, int* warnings) {
    RCP_TRY(require_ready());
    if (mem != RCP_MEM_HOST && mem != RCP_MEM_DEVICE) return fail(RCP_ERR_ARG, "kmeans: bad mem kind");
    if (algorithm != RCP_KMEANS_HARTIGAN_WONG && algorithm != RCP_KMEANS_LLOYD && algorithm != RCP_KMEANS_MACQUEEN)
        return fail(RCP_ERR_ARG, "kmeans: 'algorithm' should be one of \"Hartigan-Wong\", \"Lloyd\", \"Forgy\", "
                                 "\"MacQueen\"");
    if (sample_kind != RCP_SAMPLE_REJECTION && sample_kind != RCP_SAMPLE_ROUNDING)
        return fail(RCP_ERR_ARG, "kmeans: unknown sample kind %d", sample_kind);
    if (k < 1) return fail(RCP_ERR_ARG, "kmeans: the number of centers must be >= 1");
    if (nstart < 1) return fail(RCP_ERR_ARG, "kmeans: 'nstart' must be >= 1");
    if (iter_max < 1) return fail(RCP_ERR_ARG, "'iter.max' must be positive");
    if (m < 0 || p < 1 || ld < m) return fail(RCP_ERR_ARG, "kmeans: bad shape or leading dimension");
    if (m < k) return fail(RCP_ERR_ARG, "more cluster centers than data points");
    if (k > KM_MAX_K) return fail(RCP_ERR_UNSUPPORTED, "kmeans: more than %d clusters", KM_MAX_K);
    if (m > 0x7fffffff) return fail(RCP_ERR_UNSUPPORTED, "kmeans: more than 2^31-1 rows");
    if (x == nullptr || cluster == nullptr || centers == nullptr || withinss == nullptr || size == nullptr ||
        totss == nullptr || iter == nullptr || ifault == nullptr || warnings == nullptr)
        return fail(RCP_ERR_ARG, "kmeans: NULL pointer");
    const int S = nstart;
    DevIn<double> dx;
    RCP_TRY(dx.init(x, (size_t)(p - 1) * (size_t)ld + (size_t)m, mem));
    const double* X = dx.ptr;

    // NA/NaN/Inf: R's .C / .Fortran refuse them
    {
        int* bad = nullptr;
        RCP_TRY(dalloc(&bad, 1));
        int h_bad = 0;
        cudaError_t e = cudaMemsetAsync(bad, 0, 4, g_ctx.stream);
        if (e == cudaSuccess) {
            km_finite_kernel<<<(unsigned)std::min<int64_t>(4096, blocks_for(m * p)), TPB, 0, g_ctx.stream>>>(
                X, m, p, ld, bad);
            g_ctx.launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream);
        dfree(bad);
        if (e != cudaSuccess) return fail(RCP_ERR_CUDA, "kmeans: finiteness check failed: %s", cudaGetErrorString(e));
        if (h_bad) return fail(RCP_ERR_DATA, "NA/NaN/Inf in foreign function call (arg 1)");
    }

    KmState st;
    st.m = m;
    st.p = p;
    st.ld = ld;
    st.k = k;
    st.S = S;
    RCP_TRY(dalloc(&st.cen, (size_t)S * k * p));
    RCP_TRY(dalloc(&st.cl, (size_t)S * m));
    RCP_TRY(dalloc(&st.nc, (size_t)S * k));
    RCP_TRY(dalloc(&st.iter, (size_t)S));
    RCP_TRY(dalloc(&st.ifault, (size_t)S));

    // ---- the initial centres, drawn as kmeans draws them
    std::unique_ptr<RRng> rng(new RRng);
    rng->seed((uint32_t)seed, sample_kind);
    std::vector<int32_t> pos((size_t)S * k);
    int32_t* d_pos = nullptr;
    int32_t* uidx = nullptr;
    RCP_TRY(dalloc(&d_pos, pos.size()));
    struct Free {
        int32_t*& a;
        int32_t*& b;
        ~Free() {
            dfree(a);
            dfree(b);
        }
    } fr{d_pos, uidx};
    const dim3 gg(blocks_for((int64_t)k * p), S);
    bool use_unique = S >= 2;
    if (S == 1) {                       // centers <- x[sample.int(m, k), ]
        r_sample_int(*rng, m, k, pos.data());
        RCP_CUDA(cudaMemcpyAsync(d_pos, pos.data(), (size_t)k * 4, cudaMemcpyHostToDevice, g_ctx.stream));
        km_gather_kernel<<<gg, TPB, 0, g_ctx.stream>>>(X, p, ld, k, d_pos, nullptr, st.cen);
        RCP_LAUNCHED();
        std::vector<double> c0((size_t)k * p);
        RCP_CUDA(cudaMemcpyAsync(c0.data(), st.cen, c0.size() * 8, cudaMemcpyDeviceToHost, g_ctx.stream));
        RCP_CUDA(cudaStreamSynchronize(g_ctx.stream));
        for (int a = 0; a < k && !use_unique; a++)          // any(duplicated(centers))
            for (int b = 0; b < a && !use_unique; b++) use_unique = rows_equal(c0.data(), c0.data(), k, p, a, b);
    }
    if (use_unique) {                   // cn <- unique(x); centers <- cn[sample.int(mm, k), ] per start
        int64_t mm = 0;
        RCP_TRY(unique_rows(X, m, p, ld, &uidx, &mm));
        if (mm < k) return fail(RCP_ERR_DATA, "more cluster centers than distinct data points.");
        for (int s = 0; s < S; s++) r_sample_int(*rng, mm, k, pos.data() + (size_t)s * k);
        RCP_CUDA(cudaMemcpyAsync(d_pos, pos.data(), pos.size() * 4, cudaMemcpyHostToDevice, g_ctx.stream));
        km_gather_kernel<<<gg, TPB, 0, g_ctx.stream>>>(X, p, ld, k, d_pos, uidx, st.cen);
        RCP_LAUNCHED();
    }

    // ---- the starts
    int alg = algorithm;
    if (k == 1) alg = RCP_KMEANS_MACQUEEN;                        // as kmeans does
    if (alg == RCP_KMEANS_HARTIGAN_WONG && k >= m)                // kmns IFAULT = 3
        return fail(RCP_ERR_DATA, "number of cluster centres must lie between 1 and nrow(x)");
    RCP_CUDA(cudaMemsetAsync(st.ifault, 0, (size_t)S * 4, g_ctx.stream));
    if (alg == RCP_KMEANS_LLOYD) {
        std::vector<int> init((size_t)S, iter_max + 1);
        RCP_CUDA(cudaMemcpyAsync(st.iter, init.data(), (size_t)S * 4, cudaMemcpyHostToDevice, g_ctx.stream));
        RCP_TRY(run_lloyd(X, st, iter_max));
    } else {
        if (alg == RCP_KMEANS_HARTIGAN_WONG) {
            RCP_TRY(dalloc(&st.ic2, (size_t)S * m));
            RCP_TRY(dalloc(&st.D, (size_t)S * m));
        }
        RCP_TRY(run_walk(X, st, iter_max, alg == RCP_KMEANS_HARTIGAN_WONG));
    }

    // ---- wss, sizes, totss; the best start
    std::vector<double> h_wss((size_t)S * k), h_colss((size_t)p);
    std::vector<int32_t> h_nc((size_t)S * k);
    std::vector<int> h_iter((size_t)S), h_fault((size_t)S);
    {
        double *e = nullptr, *wss = nullptr, *colss = nullptr;
        RCP_TRY(dalloc(&e, (size_t)S * m));
        RCP_TRY(dalloc(&wss, (size_t)S * k));
        RCP_TRY(dalloc(&colss, (size_t)p));
        km_err_kernel<<<dim3(blocks_for(m), S), TPB, 0, g_ctx.stream>>>(X, m, p, ld, k, st.cen, st.cl, e);
        km_wss_kernel<<<dim3(k, S), TPB, 0, g_ctx.stream>>>(m, k, st.cl, e, wss, st.nc);
        km_colss_kernel<<<(unsigned)p, TPB, 0, g_ctx.stream>>>(X, m, ld, colss);
        g_ctx.launches += 3;
        cudaError_t ce = cudaGetLastError();
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(h_wss.data(), wss, h_wss.size() * 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(h_colss.data(), colss, h_colss.size() * 8, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(h_nc.data(), st.nc, h_nc.size() * 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(h_iter.data(), st.iter, (size_t)S * 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(h_fault.data(), st.ifault, (size_t)S * 4, cudaMemcpyDeviceToHost, g_ctx.stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(g_ctx.stream);
        dfree(e);
        dfree(wss);
        dfree(colss);
        if (ce != cudaSuccess) return fail(RCP_ERR_CUDA, "kmeans failed: %s", cudaGetErrorString(ce));
    }
    int warn = 0, best = 0;
    long double best_tot = 0.0L;
    for (int s = 0; s < S; s++) {
        if (h_fault[s] == 1) return fail(RCP_ERR_DATA, "empty cluster: try a better set of initial centers");
        if (h_iter[s] > iter_max) {
            warn |= RCP_KMEANS_WARN_NOT_CONVERGED;
            h_fault[s] = 2;
        }
        if (h_fault[s] == 4) warn |= RCP_KMEANS_WARN_QUICK_TRANSFER;
        long double tot = 0.0L;
        for (int l = 0; l < k; l++) {
            tot += h_wss[(size_t)s * k + l];
            if (alg != RCP_KMEANS_HARTIGAN_WONG && h_nc[(size_t)s * k + l] == 0) warn |= RCP_KMEANS_WARN_EMPTY_CLUSTER;
        }
        const double t = (double)tot;                 // R's sum(): long double, returned as double
        if (s == 0 || t < (double)best_tot) {
            best = s;
            best_tot = t;
        }
    }
    long double tss = 0.0L;
    for (int64_t j = 0; j < p; j++) tss += h_colss[(size_t)j];
    *totss = (double)tss;
    *iter = h_iter[best];
    *ifault = h_fault[best];
    *warnings = warn;

    // ---- outputs of the best start
    const cudaMemcpyKind d2o = mem == RCP_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    const cudaMemcpyKind h2o = mem == RCP_MEM_HOST ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice;
    int32_t* d_cluster = nullptr;
    if (mem == RCP_MEM_HOST)
        RCP_TRY(dalloc(&d_cluster, (size_t)m));
    else
        d_cluster = cluster;
    km_cluster_out_kernel<<<blocks_for(m), TPB, 0, g_ctx.stream>>>(m, st.cl + (int64_t)best * m, d_cluster);
    g_ctx.launches++;
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess && mem == RCP_MEM_HOST)
        ce = cudaMemcpyAsync(cluster, d_cluster, (size_t)m * 4, cudaMemcpyDeviceToHost, g_ctx.stream);
    if (ce == cudaSuccess)
        ce = cudaMemcpyAsync(centers, st.cen + (int64_t)best * k * p, (size_t)k * p * 8, d2o, g_ctx.stream);
    if (ce == cudaSuccess)
        ce = cudaMemcpyAsync(withinss, h_wss.data() + (size_t)best * k, (size_t)k * 8, h2o, g_ctx.stream);
    if (ce == cudaSuccess)
        ce = cudaMemcpyAsync(size, h_nc.data() + (size_t)best * k, (size_t)k * 4, h2o, g_ctx.stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(g_ctx.stream);
    if (mem == RCP_MEM_HOST) dfree(d_cluster);
    if (ce != cudaSuccess) return fail(RCP_ERR_CUDA, "kmeans: copy of the results failed: %s", cudaGetErrorString(ce));
    return RCP_OK;
}
