/*
 * csr_twin.c -- CPU twin of KL_OP_CSR and of KL_PC_JACOBI_CHEB on it (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * Definition (ours; the GPU kernels k_csr_spmv and k_csr_jacobi_cheb_step in kl_csr.cu are held to it bit for bit):
 *   W = the smallest power of two >= ceil(nnz / n), clamped to [1, 32]
 *   row i, lane l < W: s_l = 0 ; s_l = fma(val[k], x[col[k]], s_l) for k = row_ptr[i] + l, + W, ... < row_ptr[i+1]
 *   butterfly: for off = W/2, ..., 1: s_l = s_l + s_(l xor off) ; y[i] = s_0
 *   diag(A): the same lanes add their diagonal entries (d_l += val[k]) and the same butterfly combines them
 *   Jacobi-Chebyshev: the arithmetic of jacobi_cheb_twin.c with dinv = 1.0 / diag(A)
 * An entry whose column is outside [0, n) contributes nothing (the kernels' guard).
 * csr_apply and csr_precond have the oracle's operator and preconditioner signatures (oracle/krylov_extras.c
 * ko_stencil_fn / ko_precond_fn), so that the oracle solvers run on the twin; the matrix comes from csr_set.
 * Built by tests/csr_twin.py with the oracle's flags (explicit fma, no contraction).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef void (*csr_stencil_fn)(const double *x, double *y, int n);

static int64_t g_n = 0, g_nnz = 0;
static const int64_t *g_rp = NULL;
static const int32_t *g_ci = NULL;
static const double *g_v = NULL;
static int g_degree = 0;

void csr_set(int64_t n, int64_t nnz, const int64_t *row_ptr, const int32_t *col_ind, const double *val)
{
    g_n = n; g_nnz = nnz; g_rp = row_ptr; g_ci = col_ind; g_v = val;
}
void csr_set_degree(int k) { g_degree = k; }

int csr_width(int64_t n, int64_t nnz)
{
    const int64_t per = n > 0 ? (nnz + n - 1) / n : 0;
    int w = 1;
    while (w < 32 && w < per) w *= 2;
    return w;
}

static void butterfly(double *s, int W)
{
    double t[32];
    for (int off = W / 2; off >= 1; off /= 2) {
        for (int l = 0; l < W; ++l) t[l] = s[l] + s[l ^ off];
        for (int l = 0; l < W; ++l) s[l] = t[l];
    }
}

/* row i of A x (dot != 0) and of diag(A) (diag != NULL) */
static double row_scan(int64_t i, int W, const double *x, double *diag)
{
    double s[32], d[32];
    int64_t lo = g_rp[i], hi = g_rp[i + 1];
    if (lo < 0) lo = 0;
    if (lo > g_nnz) lo = g_nnz;
    if (hi > g_nnz) hi = g_nnz;
    for (int l = 0; l < W; ++l) {
        s[l] = 0.0;
        d[l] = 0.0;
        for (int64_t k = lo + l; k < hi; k += W) {
            const int32_t c = g_ci[k];
            if ((uint32_t)c >= (uint32_t)g_n) continue;
            if (x) s[l] = fma(g_v[k], x[c], s[l]);
            if (c == i) d[l] += g_v[k];
        }
    }
    butterfly(s, W);
    if (diag) {
        butterfly(d, W);
        *diag = d[0];
    }
    return s[0];
}

void csr_spmv(const double *x, double *y)
{
    const int W = csr_width(g_n, g_nnz);
#pragma omp for
    for (int64_t i = 0; i < g_n; ++i) y[i] = row_scan(i, W, x, NULL);
}

void csr_diag(double *diag)
{
    const int W = csr_width(g_n, g_nnz);
#pragma omp for
    for (int64_t i = 0; i < g_n; ++i) row_scan(i, W, NULL, diag + i);
}

/* the oracle's stencil signature; n (the grid extent) is ignored, the matrix is the one set by csr_set */
void csr_apply(const double *x, double *y, int n_unused)
{
    (void)n_unused;
    csr_spmv(x, y);
}

/* z = M^-1 r; needs one scratch vector (aux, holds A z); d and dinv are allocated here.  Callable inside or outside an
 * OpenMP parallel region (orphaned work-sharing, like the oracle's preconditioners). */
void csr_jacobi_cheb(const double *r, double *z, double *aux, const double *params)
{
    static double *buf = NULL;
    static int64_t blen = 0;
    const int64_t len = g_n;
#pragma omp single
    {
        if (blen < len) { free(buf); buf = malloc(sizeof(double) * 2 * len); blen = len; }
    }
    double *dinv = buf, *d = buf + len;
    csr_diag(dinv);
#pragma omp for
    for (int64_t i = 0; i < len; ++i) dinv[i] = 1.0 / dinv[i];
    if (g_degree == 0) {
#pragma omp for
        for (int64_t i = 0; i < len; ++i) z[i] = r[i] * dinv[i];
        return;
    }
    double ea = params[0], eb = params[1];
    double theta = (eb + ea) / 2.0, delta = fabs(eb - ea) / 2.0;
    double sigma = theta / delta, rho_prev = 1.0 / sigma;
#pragma omp for
    for (int64_t i = 0; i < len; ++i) { d[i] = (r[i] * dinv[i]) / theta; z[i] = d[i]; }
    for (int k = 0; k < g_degree; ++k) {
        double rho = 1.0 / (2.0 * sigma - rho_prev);
        double c1 = rho * rho_prev, c2 = 2.0 * rho / delta;
        csr_spmv(z, aux);
#pragma omp for
        for (int64_t i = 0; i < len; ++i) {
            d[i] = fma(c1, d[i], c2 * ((r[i] - aux[i]) * dinv[i]));
            z[i] = z[i] + d[i];
        }
        rho_prev = rho;
    }
}

/* the oracle's preconditioner signature (A_x is not used: the operator is the twin's own) */
void csr_precond(csr_stencil_fn A_x, const double *r, double *z, double *aux, const double *params, int n, int64_t len)
{
    (void)A_x;
    (void)n;
    (void)len;
    csr_jacobi_cheb(r, z, aux, params);
}
