/* ORACLE (test infrastructure, never linked into the product): hclust(dist(x), "complete") of
 * stats, restated in plain C.  Parity unpinned: R's sources are not vendored; this restates
 *   - R_euclidean of distance.c (no NA branch: non-finite input is refused by the caller),
 *   - hclust.f (F. Murtagh, as R ships it) for iOpt = 3, complete linkage, and
 *   - HCASS2 of the same file, its literal O(n^2) loops,
 * in their order of operations.  Built with -ffp-contract=off (oracle/cbuild.py); OpenMP, where
 * available, splits the distance columns only, which cannot change a bit. */
#include <math.h>
#include <stdint.h>

#define INF 1e300

/* dist(x): column-major n x p x with leading dimension ld -> the lower triangle by columns, as R's
 * "dist" object stores it: d[(j, i)] for j < i at IOFFST(n, j, i). */
static int64_t ioffst(int64_t n, int64_t i, int64_t j) /* 1-based, i < j */
{
    return j + (i - 1) * n - (i * (i + 1)) / 2;
}

void ohc_dist(const double* x, int64_t n, int64_t p, int64_t ld, double* d)
{
    int64_t j;
#pragma omp parallel for schedule(dynamic, 16)
    for (j = 0; j < n; j++) {
        int64_t at = ioffst(n, j + 1, j + 2) - 1;
        for (int64_t i = j + 1; i < n; i++) {
            double dist = 0.0;
            for (int64_t c = 0; c < p; c++) {
                double dev = x[i + c * ld] - x[j + c * ld];
                dist += dev * dev;
            }
            d[at++] = sqrt(dist);
        }
    }
}

/* hclust.f, iOpt = 3.  diss (condensed, overwritten), 1-based ia / ib / crit of n - 1 merges;
 * nn (int n), disnn (double n), flag (char n) are work arrays.  Returns 0, or 1 when a distance
 * reached INF. */
int ohc_hclust(int n, double* diss, int* ia, int* ib, double* crit, int* nn, double* disnn, char* flag)
{
    int i, j, k, im = 0, jm = 0, jj = 0, i2, j2, ncl;
    double dmin;
#define DISS(a) diss[(a) - 1]
#define NN(a) nn[(a) - 1]
#define DISNN(a) disnn[(a) - 1]
#define FLAG(a) flag[(a) - 1]
    for (i = 1; i <= n; i++) FLAG(i) = 1;
    ncl = n;
    /* the list of nearest neighbours to the right */
    for (i = 1; i <= n - 1; i++) {
        dmin = INF;
        for (j = i + 1; j <= n; j++) {
            int64_t ind = ioffst(n, i, j);
            if (dmin > DISS(ind)) {
                dmin = DISS(ind);
                jm = j;
            }
        }
        if (dmin >= INF) return 1;
        NN(i) = jm;
        DISNN(i) = dmin;
    }
    while (ncl > 1) {
        /* the least dissimilarity from the list of NNs */
        dmin = INF;
        for (i = 1; i <= n - 1; i++)
            if (FLAG(i) && DISNN(i) < dmin) {
                dmin = DISNN(i);
                im = i;
                jm = NN(i);
            }
        ncl--;
        i2 = im < jm ? im : jm;
        j2 = im < jm ? jm : im;
        ia[n - ncl - 1] = i2;
        ib[n - ncl - 1] = j2;
        crit[n - ncl - 1] = dmin;
        FLAG(j2) = 0;
        /* the dissimilarities from the new cluster */
        dmin = INF;
        for (k = 1; k <= n; k++) {
            if (FLAG(k) && k != i2) {
                int64_t ind1 = i2 < k ? ioffst(n, i2, k) : ioffst(n, k, i2);
                int64_t ind2 = j2 < k ? ioffst(n, j2, k) : ioffst(n, k, j2);
                DISS(ind1) = DISS(ind1) > DISS(ind2) ? DISS(ind1) : DISS(ind2);   /* MAX */
                if (i2 < k) {
                    if (DISS(ind1) < dmin) {
                        dmin = DISS(ind1);
                        jj = k;
                    }
                } else if (DISS(ind1) < DISNN(k)) {   /* k < i2: JB's fix */
                    DISNN(k) = DISS(ind1);
                    NN(k) = i2;
                }
            }
        }
        DISNN(i2) = dmin;
        NN(i2) = jj;
        /* the NNs that pointed at i2 or j2 */
        for (i = 1; i <= n - 1; i++) {
            if (FLAG(i) && (NN(i) == i2 || NN(i) == j2)) {
                dmin = INF;
                for (j = i + 1; j <= n; j++) {
                    if (FLAG(j)) {
                        int64_t ind = ioffst(n, i, j);
                        if (DISS(ind) < dmin) {
                            dmin = DISS(ind);
                            jj = j;
                        }
                    }
                }
                NN(i) = jj;
                DISNN(i) = dmin;
            }
        }
    }
    return 0;
#undef DISS
#undef NN
#undef DISNN
#undef FLAG
}

/* HCASS2: 1-based ia / ib (n - 1 each) -> iia / iib (R's merge columns) and iorder (1-based). */
void ohc_hcass2(int n, const int* ia, const int* ib, int* iorder, int* iia, int* iib)
{
    int i, j, k, k1, k2, loc;
    for (i = 0; i < n; i++) {
        iia[i] = i < n - 1 ? ia[i] : 0;
        iib[i] = i < n - 1 ? ib[i] : 0;
    }
    for (i = 1; i <= n - 2; i++) {
        k = ia[i - 1] < ib[i - 1] ? ia[i - 1] : ib[i - 1];
        for (j = i + 1; j <= n - 1; j++) {
            if (ia[j - 1] == k) iia[j - 1] = -i;
            if (ib[j - 1] == k) iib[j - 1] = -i;
        }
    }
    for (i = 1; i <= n - 1; i++) {
        iia[i - 1] = -iia[i - 1];
        iib[i - 1] = -iib[i - 1];
    }
    for (i = 1; i <= n - 1; i++) {
        if (iia[i - 1] > 0 && iib[i - 1] < 0) {
            k = iia[i - 1];
            iia[i - 1] = iib[i - 1];
            iib[i - 1] = k;
        }
        if (iia[i - 1] > 0 && iib[i - 1] > 0) {
            k1 = iia[i - 1] < iib[i - 1] ? iia[i - 1] : iib[i - 1];
            k2 = iia[i - 1] < iib[i - 1] ? iib[i - 1] : iia[i - 1];
            iia[i - 1] = k1;
            iib[i - 1] = k2;
        }
    }
    /* the order: expand the clusters from the last merge down */
    iorder[0] = iia[n - 2];
    iorder[1] = iib[n - 2];
    loc = 2;
    for (i = n - 2; i >= 1; i--) {
        for (j = 1; j <= loc; j++) {
            if (iorder[j - 1] == i) {
                iorder[j - 1] = iia[i - 1];
                if (j == loc) {
                    loc++;
                    iorder[loc - 1] = iib[i - 1];
                } else {
                    loc++;
                    for (k = loc; k >= j + 2; k--) iorder[k - 1] = iorder[k - 2];
                    iorder[j] = iib[i - 1];
                }
                break;
            }
        }
    }
    for (i = 1; i <= n; i++) iorder[i - 1] = -iorder[i - 1];
}
