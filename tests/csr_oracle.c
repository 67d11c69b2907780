/*
 * csr_oracle.c -- CPU oracle of CSR storage, O(nnz) per mat-vec.  TEST INFRASTRUCTURE ONLY:
 * compiled by tests/csr_oracle.py into a temporary directory, never linked into the product.
 *
 * It includes the dense oracle's source unchanged, so the chunk256 / det_sum reductions and the
 * lane-order butterfly are literally the dense oracle's; only the mat-vec touches the stored
 * entries instead of every column.  A lane-order accumulator is never -0 (it starts at +0 and an
 * exactly-zero sum rounds to +0 unless both operands are -0), so a zero entry leaves it unchanged
 * for finite p: every result equals cgo_solve on the densified matrix bit for bit, which
 * tests/test_sparse_cpu.py checks.
 *
 * CSR of rows [row0, row0 + rows): rp[rows + 1] int64, col int32 (ascending, unique per row), val.
 */
#include "../oracle/cg_oracle.c"

#include <stdint.h>

/* generate_lap2d_matrix's non-zeros (cg.cc:159-188) of rows [row0, row0+nrows), ascending
 * columns; returns nnz.  col == NULL: count only (rp, when given, still filled). */
int64_t cso_generate_lap2d(int64_t n, int64_t row0, int64_t nrows, int64_t *rp, int32_t *col, double *val)
{
    int64_t inc = (int64_t)floor(sqrt((double)n));
    int64_t k = 0;
    for (int64_t li = 0; li < nrows; ++li) {
        int64_t i = row0 + li;
        int64_t c[5];
        double v[5];
        int m = 0;
        if (i > inc) { c[m] = i - 1 - inc; v[m++] = -1.0; }
        if (i > 0) { c[m] = i - 1; v[m++] = -1.0; }
        c[m] = i; v[m++] = 4.0;
        if (i < n - 1) { c[m] = i + 1; v[m++] = -1.0; }
        if (i < n - 1 - inc) { c[m] = i + 1 + inc; v[m++] = -1.0; }
        if (rp) rp[li] = k;
        for (int e = 0; e < m; ++e, ++k)
            if (col) {
                col[k] = (int32_t)c[e];
                val[k] = v[e];
            }
    }
    if (rp) rp[nrows] = k;
    return k;
}

/* lane order over the stored entries: bucket c % 64 is the fma chain over its entries in
 * ascending column order from +0, then the dense oracle's lane sum and butterfly */
double cso_row_dot(const int32_t *col, const double *val, int64_t len, const double *p)
{
    double acc[64];
    for (int j = 0; j < 64; ++j) acc[j] = 0.0;
    for (int64_t k = 0; k < len; ++k) acc[col[k] & 63] = fma(val[k], p[col[k]], acc[col[k] & 63]);
    double lane[32];
    for (int l = 0; l < 32; ++l) lane[l] = acc[2 * l] + acc[2 * l + 1];
    return butterfly32(lane);
}

void cso_gemv(int64_t rows, const int64_t *rp, const int32_t *col, const double *val, const double *p, double *y)
{
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < rows; ++i) y[i] = cso_row_dot(col + rp[i], val + rp[i], rp[i + 1] - rp[i], p);
}

/* cgo_residual_check with the CSR mat-vec */
void cso_residual_check(int64_t n, const int64_t *rp, const int32_t *col, const double *val, const double *b,
                        const double *x, double *norm_x, double *rel_resid)
{
    double *r = (double *)malloc(sizeof(double) * (size_t)n);
    cso_gemv(n, rp, col, val, x, r);
    for (int64_t i = 0; i < n; ++i) r[i] = fma(-1.0, b[i], r[i]);
    *rel_resid = sqrt(cgo_dot(r, r, n)) / sqrt(cgo_dot(b, b, n));
    *norm_x = sqrt(cgo_dot(x, x, n));
    free(r);
}

/* cgo_solve (cg.cc:38-156) with the CSR mat-vec: the same statements in the same order */
void cso_solve(int64_t n, const int64_t *rp, const int32_t *col, const double *val, const double *b, double *x,
               int64_t max_iter, double tol, double *hist, cgo_info *info)
{
    double *r = (double *)malloc(sizeof(double) * (size_t)n);
    double *p = (double *)malloc(sizeof(double) * (size_t)n);
    double *Ap = (double *)malloc(sizeof(double) * (size_t)n);

    cso_gemv(n, rp, col, val, x, Ap);                                  /* cg.cc:77-82 */
    for (int64_t i = 0; i < n; ++i) r[i] = fma(-1.0, Ap[i], b[i]);
    memcpy(p, r, sizeof(double) * (size_t)n);                          /* :85-88 */
    double rsold = cgo_dot(r, p, n);                                   /* :91-92 */
    double rsnew = rsold;
    int converged = 0;

    int64_t k = 0;
    for (; k < max_iter; ++k) {
        cso_gemv(n, rp, col, val, p, Ap);                              /* :100-102 */
        double conj = cgo_dot(p, Ap, n);                               /* :105-106 */
        double clamp = rsold * NEARZERO;
        double alpha = rsold / ((conj < clamp) ? clamp : conj);        /* :107 */
        for (int64_t i = 0; i < n; ++i) x[i] = fma(alpha, p[i], x[i]); /* :110 */
        double nalpha = -alpha;
        for (int64_t i = 0; i < n; ++i) r[i] = fma(nalpha, Ap[i], r[i]); /* :113 */
        rsnew = cgo_dot(r, r, n);                                      /* :116-117 */
        if (hist) hist[k] = rsnew;
        if (sqrt(rsnew) < tol) { converged = 1; break; }               /* :120-121 */
        double beta = rsnew / rsold;                                   /* :124 */
        for (int64_t i = 0; i < n; ++i) p[i] = fma(beta, p[i], r[i]);  /* :127-129 */
        rsold = rsnew;                                                 /* :132 */
    }

    if (info) {
        info->k = k;
        info->converged = converged;
        info->rsold = rsold;
        info->rsnew = rsnew;
        cso_residual_check(n, rp, col, val, b, x, &info->norm_x, &info->rel_resid);
    }
    free(r); free(p); free(Ap);
}
