/* ORACLE (test infrastructure, never linked into the product): plain C restatement of the three
 * algorithms of stats::kmeans -- kmeans_Lloyd and kmeans_MacQueen (R src/library/stats/src/
 * kmeans.c) and AS 136 as R ships it (kmns.f: KMNS, OPTRA, QTRAN).  Parity unpinned: R's sources
 * are not vendored; this follows the published algorithms and R's documented loops.
 *
 * Built with -ffp-contract=off, as x86-64 builds of R are: every distance is
 * tmp = x - c; dd += tmp * tmp, columns in order, and no product is fused into an add.
 * x: column-major m x p with leading dimension ld; cen: column-major k x p (in: the initial
 * centres, out: the final ones); cl: 1-based; *iter: in iter.max, out as R reports it. */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define X(i, j) x[(int64_t)(i) + (int64_t)(j) * ld]
#define CEN(l, j) cen[(int64_t)(l) + (int64_t)(j) * k]

static double dist(const double* x, int64_t ld, int64_t p, const double* cen, int k, int64_t i, int l) {
    double dd = 0.0;
    for (int64_t c = 0; c < p; c++) {
        const double tmp = X(i, c) - CEN(l, c);
        dd += tmp * tmp;
    }
    return dd;
}

static void means(const double* x, int64_t m, int64_t p, int64_t ld, double* cen, int k, const int32_t* cl,
                  int32_t* nc) {
    for (int64_t j = 0; j < (int64_t)k * p; j++) cen[j] = 0.0;
    for (int j = 0; j < k; j++) nc[j] = 0;
    for (int64_t i = 0; i < m; i++) {
        const int it = cl[i] - 1;
        nc[it]++;
        for (int64_t c = 0; c < p; c++) CEN(it, c) += X(i, c);
    }
    for (int64_t j = 0; j < (int64_t)k * p; j++) cen[j] /= nc[j % k];
}

static void wss_rows(const double* x, int64_t m, int64_t p, int64_t ld, const double* cen, int k,
                     const int32_t* cl, double* wss) {
    for (int j = 0; j < k; j++) wss[j] = 0.0;
    for (int64_t i = 0; i < m; i++) {
        const int it = cl[i] - 1;
        for (int64_t c = 0; c < p; c++) {
            const double tmp = X(i, c) - CEN(it, c);
            wss[it] += tmp * tmp;
        }
    }
}

void okm_lloyd(const double* x, int64_t m, int64_t p, int64_t ld, double* cen, int k, int32_t* cl, int* piter,
               int32_t* nc, double* wss) {
    const int maxiter = *piter;
    int iter, inew = 0;
    for (int64_t i = 0; i < m; i++) cl[i] = -1;
    for (iter = 0; iter < maxiter; iter++) {
        int updated = 0;
        for (int64_t i = 0; i < m; i++) {
            double best = INFINITY;
            for (int j = 0; j < k; j++) {
                const double dd = dist(x, ld, p, cen, k, i, j);
                if (dd < best) {
                    best = dd;
                    inew = j + 1;
                }
            }
            if (cl[i] != inew) {
                updated = 1;
                cl[i] = inew;
            }
        }
        if (!updated) break;
        means(x, m, p, ld, cen, k, cl, nc);
    }
    *piter = iter + 1;
    wss_rows(x, m, p, ld, cen, k, cl, wss);
}

void okm_macqueen(const double* x, int64_t m, int64_t p, int64_t ld, double* cen, int k, int32_t* cl, int* piter,
                  int32_t* nc, double* wss) {
    const int maxiter = *piter;
    int iter, inew = 0;
    for (int64_t i = 0; i < m; i++) {
        double best = INFINITY;
        for (int j = 0; j < k; j++) {
            const double dd = dist(x, ld, p, cen, k, i, j);
            if (dd < best) {
                best = dd;
                inew = j + 1;
            }
        }
        cl[i] = inew;
    }
    means(x, m, p, ld, cen, k, cl, nc);
    for (iter = 0; iter < maxiter; iter++) {
        int updated = 0;
        for (int64_t i = 0; i < m; i++) {
            double best = INFINITY;
            for (int j = 0; j < k; j++) {
                const double dd = dist(x, ld, p, cen, k, i, j);
                if (dd < best) {
                    best = dd;
                    inew = j;
                }
            }
            const int iold = cl[i] - 1;
            if (iold != inew) {
                updated = 1;
                cl[i] = inew + 1;
                nc[iold]--;
                nc[inew]++;
                for (int64_t c = 0; c < p; c++) {
                    CEN(iold, c) += (CEN(iold, c) - X(i, c)) / nc[iold];
                    CEN(inew, c) += (X(i, c) - CEN(inew, c)) / nc[inew];
                }
            }
        }
        if (!updated) break;
    }
    *piter = iter + 1;
    wss_rows(x, m, p, ld, cen, k, cl, wss);
}

/* ---- AS 136 ------------------------------------------------------------------------------ */
#define BIG 1.0e30

typedef struct {
    const double* x;
    int64_t m, p, ld;
    double* cen;
    int k;
    int32_t *ic1, *ic2, *nc, *itran;
    double *an1, *an2, *d;
    int64_t *ncp, *live;
} Hw;

static double hw_d(const Hw* h, int64_t i, int l) { return dist(h->x, h->ld, h->p, h->cen, h->k, i, l); }

static void hw_transfer(Hw* h, int64_t i, int l1, int l2) {
    const double* x = h->x;
    const int64_t ld = h->ld;
    double* cen = h->cen;
    const int k = h->k;
    const double al1 = h->nc[l1], alw = al1 - 1.0, al2 = h->nc[l2], alt = al2 + 1.0;
    for (int64_t j = 0; j < h->p; j++) {
        CEN(l1, j) = (CEN(l1, j) * al1 - X(i, j)) / alw;
        CEN(l2, j) = (CEN(l2, j) * al2 + X(i, j)) / alt;
    }
    h->nc[l1]--;
    h->nc[l2]++;
    h->an2[l1] = alw / al1;
    h->an1[l1] = BIG;
    if (alw > 1.0) h->an1[l1] = alw / (alw - 1.0);
    h->an1[l2] = alt / al2;
    h->an2[l2] = alt / (alt + 1.0);
    h->ic1[i] = l2;
    h->ic2[i] = l1;
}

static void optra(Hw* h, int64_t* indx) {
    const int k = h->k;
    const int64_t m = h->m;
    for (int l = 0; l < k; l++)
        if (h->itran[l] == 1) h->live[l] = m + 1;
    for (int64_t i = 0; i < m; i++) {
        const int64_t i1 = i + 1;
        (*indx)++;
        const int l1 = h->ic1[i];
        if (h->nc[l1] != 1) {
            if (h->ncp[l1] != 0) h->d[i] = hw_d(h, i, l1) * h->an1[l1];
            int l2 = h->ic2[i];
            const int ll = l2;
            double r2 = hw_d(h, i, l2) * h->an2[l2];
            for (int l = 0; l < k; l++) {
                if ((i1 >= h->live[l1] && i1 >= h->live[l]) || l == l1 || l == ll) continue;
                const double rr = r2 / h->an2[l];
                const double dc = hw_d(h, i, l);    /* kmns.f exits the sum at DC >= RR: same decision */
                if (dc < rr) {
                    r2 = dc * h->an2[l];
                    l2 = l;
                }
            }
            if (r2 >= h->d[i]) {
                h->ic2[i] = l2;
            } else {
                *indx = 0;
                h->live[l1] = m + i1;
                h->live[l2] = m + i1;
                h->ncp[l1] = i1;
                h->ncp[l2] = i1;
                hw_transfer(h, i, l1, l2);
            }
        }
        if (*indx == m) return;
    }
    for (int l = 0; l < k; l++) {
        h->itran[l] = 0;
        h->live[l] -= m;
    }
}

/* returns 1 when the step limit was reached */
static int qtran(Hw* h, int64_t* indx, int64_t imaxqtr) {
    const int64_t m = h->m;
    int64_t icoun = 0, istep = 0;
    for (;;) {
        for (int64_t i = 0; i < m; i++) {
            icoun++;
            istep++;
            if (istep >= imaxqtr) return 1;
            const int l1 = h->ic1[i], l2 = h->ic2[i];
            if (h->nc[l1] != 1) {
                if (istep <= h->ncp[l1]) h->d[i] = hw_d(h, i, l1) * h->an1[l1];
                if (istep < h->ncp[l1] || istep < h->ncp[l2]) {
                    const double r2 = h->d[i] / h->an2[l2];
                    if (hw_d(h, i, l2) < r2) {
                        icoun = 0;
                        *indx = 0;
                        h->itran[l1] = 1;
                        h->itran[l2] = 1;
                        h->ncp[l1] = istep + m;
                        h->ncp[l2] = istep + m;
                        hw_transfer(h, i, l1, l2);
                    }
                }
            }
            if (icoun == m) return 0;
        }
    }
}

/* kmns: ifault 0, 1 (empty cluster after the first assignment), 2 (iter.max reached), 3 (k <= 1
 * or k >= m), 4 (quick-transfer step limit).  work: 4 m int32 + m double + 6 k doubles/ints are
 * allocated by the caller through the arrays below. */
void okm_hartigan_wong(const double* x, int64_t m, int64_t p, int64_t ld, double* cen, int k, int32_t* cl,
                       int* piter, int32_t* nc, double* wss, int* ifault, int32_t* ic2, double* d, double* an1,
                       double* an2, int32_t* itran, int64_t* ncp, int64_t* live) {
    Hw h = {x, m, p, ld, cen, k, cl, ic2, nc, itran, an1, an2, d, ncp, live};
    const int maxiter = *piter;
    *ifault = 3;
    if (k <= 1 || k >= m) return;
    for (int64_t i = 0; i < m; i++) {
        int c1 = 0, c2 = 1;
        double dt1 = hw_d(&h, i, 0), dt2 = hw_d(&h, i, 1);
        if (dt1 > dt2) {
            c1 = 1;
            c2 = 0;
            const double t = dt1;
            dt1 = dt2;
            dt2 = t;
        }
        for (int l = 2; l < k; l++) {
            const double db = hw_d(&h, i, l);
            if (db >= dt2) continue;
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
        cl[i] = c1;
        ic2[i] = c2;
    }
    for (int64_t j = 0; j < (int64_t)k * p; j++) cen[j] = 0.0;
    for (int l = 0; l < k; l++) nc[l] = 0;
    for (int64_t i = 0; i < m; i++) {
        nc[cl[i]]++;
        for (int64_t j = 0; j < p; j++) CEN(cl[i], j) += X(i, j);
    }
    *ifault = 1;
    for (int l = 0; l < k; l++)
        if (nc[l] == 0) {
            for (int64_t i = 0; i < m; i++) cl[i] += 1;
            return;
        }
    *ifault = 0;
    for (int l = 0; l < k; l++) {
        const double aa = nc[l];
        for (int64_t j = 0; j < p; j++) CEN(l, j) /= aa;
        an2[l] = aa / (aa + 1.0);
        an1[l] = BIG;
        if (aa > 1.0) an1[l] = aa / (aa - 1.0);
        itran[l] = 1;
        ncp[l] = -1;
    }
    for (int64_t i = 0; i < m; i++) d[i] = 0.0;
    int64_t indx = 0;
    const int64_t imaxqtr = 50 * m < 0x7fffffff ? 50 * m : 0x7fffffff;
    int ij, iter_out = -1;
    for (ij = 1; ij <= maxiter; ij++) {
        optra(&h, &indx);
        if (indx == m) {
            iter_out = ij;
            break;
        }
        if (qtran(&h, &indx, imaxqtr)) {
            *ifault = 4;
            iter_out = ij;
            break;
        }
        if (k == 2) {
            iter_out = ij;
            break;
        }
        for (int l = 0; l < k; l++) ncp[l] = 0;
    }
    if (iter_out < 0) {
        iter_out = maxiter + 1;
        *ifault = 2;
    }
    *piter = iter_out;
    /* the centres from scratch, then WSS (column by column, as kmns.f sums it) */
    for (int l = 0; l < k; l++) wss[l] = 0.0;
    for (int64_t j = 0; j < (int64_t)k * p; j++) cen[j] = 0.0;
    for (int64_t i = 0; i < m; i++)
        for (int64_t j = 0; j < p; j++) CEN(cl[i], j) += X(i, j);
    for (int64_t j = 0; j < p; j++) {
        for (int l = 0; l < k; l++) CEN(l, j) /= (double)nc[l];
        for (int64_t i = 0; i < m; i++) {
            const double da = X(i, j) - CEN(cl[i], j);
            wss[cl[i]] += da * da;
        }
    }
    for (int64_t i = 0; i < m; i++) cl[i] += 1;
}
