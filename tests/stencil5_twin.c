/*
 * stencil5_twin.c -- CPU twin of KL_OP_STENCIL5 (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * Definition (ours; the GPU kernels apply5 / apply5c / apply5_rt are held to it bit for bit), zero Dirichlet:
 *   y = c xc - (wl xl + wr xr + wd xd + wu xu)
 * evaluation order (shared with the CUDA kernels; the same as oracle/krylov_extras.c ko_aniso_var):
 *   s = fma(wl, xl, wr*xr) ; t = fma(wd, xd, wu*xu) ; y = fma(c, xc, -(s + t))
 * missing neighbours count as 0.  ("d" = idx+n, "u" = idx-n, the reference's naming in poisson.f90:42.)
 * s5_apply has the oracle's stencil signature (oracle/krylov_extras.c ko_stencil_fn, square grids), so the oracle
 * solvers and ko_cheb / cbpr2 run with it; s5_apply_xy takes rectangular grids.
 * Built by tests/stencil5_twin.py with the oracle's flags (explicit fma, no contraction).
 */
#include <math.h>
#include <stdint.h>

static double g_c = 4.0, g_wl = 1.0, g_wr = 1.0, g_wd = 1.0, g_wu = 1.0;
void s5_set(double c, double wl, double wr, double wd, double wu)
{
    g_c = c; g_wl = wl; g_wr = wr; g_wd = wd; g_wu = wu;
}

void s5_apply_xy(const double *x, double *y, int nx, int ny)
{
    const int64_t NX = nx, NY = ny;
    const double c = g_c, wl = g_wl, wr = g_wr, wd = g_wd, wu = g_wu;
#pragma omp for collapse(2)
    for (int64_t j = 0; j < NY; ++j)
        for (int64_t i = 0; i < NX; ++i) {
            int64_t idx = i + j * NX;
            double xl = i > 0 ? x[idx - 1] : 0.0, xr = i < NX - 1 ? x[idx + 1] : 0.0;
            double xd = j < NY - 1 ? x[idx + NX] : 0.0, xu = j > 0 ? x[idx - NX] : 0.0;
            double s = fma(wl, xl, wr * xr), t = fma(wd, xd, wu * xu);
            y[idx] = fma(c, x[idx], -(s + t));
        }
}

void s5_apply(const double *x, double *y, int n) { s5_apply_xy(x, y, n, n); }
