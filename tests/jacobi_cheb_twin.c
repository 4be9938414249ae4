/*
 * jacobi_cheb_twin.c -- CPU twin of KL_PC_JACOBI_CHEB (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * Definition (ours; the GPU kernels ChJacCheb and k_jacobi_cheb_step are held to it bit for bit):
 * Saad Alg. 12.1 on D^-1 A z = D^-1 r, A = the variable-coefficient operator of oracle/krylov_extras.c ko_aniso_var
 * on an nx x ny grid, D = diag(A).
 *   diag = ((wl + wr) + wd) + wu  (face weights exactly as in ko_aniso_var) ; dinv = 1.0/diag ; s = r*dinv
 *   degree 0: z = s (params ignored)
 *   degree k >= 1: theta, delta, sigma, rho and c1, c2 as in ko_cheb ;  d = s/theta ; z = d
 *                  for each step: d = fma(c1, d, c2*((r - A z)*dinv)) ; z = z + d
 * The spectrum of D^-1 A lies in (0, 2] (Gershgorin), so params = (a, b) is an interval inside it, in either order.
 * Built by tests/jacobi_cheb_twin.py with the oracle's flags (explicit fma, no contraction).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef void (*jc_stencil_fn)(const double *x, double *y, int n);

static const double *g_kx = NULL, *g_ky = NULL;
void jc_set_fields(const double *kx, const double *ky) { g_kx = kx; g_ky = ky; }

/* y = A(kx, ky) x ; ko_aniso_var's formula with separate extents */
void jc_aniso_var_xy(const double *x, double *y, int nx, int ny)
{
    const int64_t NX = nx, NY = ny;
    const double *kx = g_kx, *ky = g_ky;
#pragma omp for collapse(2)
    for (int64_t j = 0; j < NY; ++j)
        for (int64_t i = 0; i < NX; ++i) {
            int64_t idx = i + j * NX;
            double kxc = kx[idx], kyc = ky[idx];
            double wl = i > 0 ? 0.5 * (kxc + kx[idx - 1]) : kxc, wr = i < NX - 1 ? 0.5 * (kxc + kx[idx + 1]) : kxc;
            double wu = j > 0 ? 0.5 * (kyc + ky[idx - NX]) : kyc, wd = j < NY - 1 ? 0.5 * (kyc + ky[idx + NX]) : kyc;
            double xl = i > 0 ? x[idx - 1] : 0.0, xr = i < NX - 1 ? x[idx + 1] : 0.0;
            double xd = j < NY - 1 ? x[idx + NX] : 0.0, xu = j > 0 ? x[idx - NX] : 0.0;
            double diag = ((wl + wr) + wd) + wu;
            double s = fma(wl, xl, wr * xr), t = fma(wd, xd, wu * xu);
            y[idx] = fma(diag, x[idx], -(s + t));
        }
}

/* dinv = 1.0 / diag(A(kx, ky)) */
void jc_dinv_xy(double *dinv, int nx, int ny)
{
    const int64_t NX = nx, NY = ny;
    const double *kx = g_kx, *ky = g_ky;
#pragma omp for collapse(2)
    for (int64_t j = 0; j < NY; ++j)
        for (int64_t i = 0; i < NX; ++i) {
            int64_t idx = i + j * NX;
            double kxc = kx[idx], kyc = ky[idx];
            double wl = i > 0 ? 0.5 * (kxc + kx[idx - 1]) : kxc, wr = i < NX - 1 ? 0.5 * (kxc + kx[idx + 1]) : kxc;
            double wu = j > 0 ? 0.5 * (kyc + ky[idx - NX]) : kyc, wd = j < NY - 1 ? 0.5 * (kyc + ky[idx + NX]) : kyc;
            dinv[idx] = 1.0 / (((wl + wr) + wd) + wu);
        }
}

static int g_degree = 0;
void jc_set_degree(int k) { g_degree = k; }

/* needs one scratch vector (aux, holds A z); d and dinv are allocated here.  Callable inside or outside an OpenMP
 * parallel region (orphaned work-sharing, like the oracle's preconditioners). */
void jc_jacobi_cheb_xy(const double *r, double *z, double *aux, const double *params, int nx, int ny)
{
    static double *buf = NULL;
    static int64_t blen = 0;
    const int64_t len = (int64_t)nx * ny;
#pragma omp single
    {
        if (blen < len) { free(buf); buf = malloc(sizeof(double) * 2 * len); blen = len; }
    }
    double *dinv = buf, *d = buf + len;
    jc_dinv_xy(dinv, nx, ny);
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
        jc_aniso_var_xy(z, aux, nx, ny);
#pragma omp for
        for (int64_t i = 0; i < len; ++i) {
            d[i] = fma(c1, d[i], c2 * ((r[i] - aux[i]) * dinv[i]));
            z[i] = z[i] + d[i];
        }
        rho_prev = rho;
    }
}

/* the oracle's preconditioner signature (oracle/krylov_extras.c ko_precond_fn), square grids: the oracle solvers
 * run with the twin through it.  The operator is the twin's own (A_x is not used). */
void jc_precond(jc_stencil_fn A_x, const double *r, double *z, double *aux, const double *params, int n, int64_t len)
{
    (void)A_x;
    (void)len;
    jc_jacobi_cheb_xy(r, z, aux, params, n, n);
}
