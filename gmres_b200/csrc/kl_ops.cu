// kl_ops.cu -- operator / preconditioner application and the public apply entry points.
#include <math.h>
#include <string.h>

#include <cmath>

#include "kl_ops.cuh"

namespace kl {

int prob_init(Prob *P, Ctx *c, const kl_operator_t *op, const kl_precond_t *pc, const double *params,
              int nparams, int nx, int ny, bool validate) {
    if (!c || !op) return KL_ERR_INVALID;
    if (op->kind == KL_OP_DENSE) {
        if (nx < 2 || ny != 1) return c->fail(KL_ERR_INVALID, "dense operator: nx = n >= 2, ny = 1");
        if (!op->user) return c->fail(KL_ERR_INVALID, "KL_OP_DENSE without a matrix");
        if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "dense operators are single-GPU only");
    } else if (op->kind == KL_OP_CSR) {
        if (nx < 2 || ny != 1) return c->fail(KL_ERR_INVALID, "KL_OP_CSR: nx = n >= 2, ny = 1");
        const kl_csr_t *m = (const kl_csr_t *)op->user;
        if (!m) return c->fail(KL_ERR_INVALID, "KL_OP_CSR without a matrix");
        if (m->nnz < 0 || !m->row_ptr || (m->nnz > 0 && (!m->col_ind || !m->val)))
            return c->fail(KL_ERR_INVALID, "KL_OP_CSR: nnz >= 0, row_ptr and (nnz > 0) col_ind and val non-null");
        if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "KL_OP_CSR is single-GPU only");
    } else if (nx < 2 || ny < 2) return c->fail(KL_ERR_INVALID, "grid must be at least 2x2");
    P->c = c;
    P->op = *op;
    P->w5 = kl_stencil5_t{0.0, 0.0, 0.0, 0.0, 0.0};
    P->csr = kl_csr_t{0, nullptr, nullptr, nullptr};
    if (pc) P->pc = *pc;
    else P->pc = kl_precond_t{KL_PC_NONE, 0, nullptr, nullptr};
    if (P->op.kind != KL_OP_POISSON5 && P->op.kind != KL_OP_POISSON5_BRANCHY && P->op.kind != KL_OP_ANISO5 &&
        P->op.kind != KL_OP_USER && P->op.kind != KL_OP_DENSE && P->op.kind != KL_OP_ANISO5_VAR &&
        P->op.kind != KL_OP_STENCIL5 && P->op.kind != KL_OP_CSR)
        return c->fail(KL_ERR_INVALID, "unknown operator kind");
    if (P->op.kind == KL_OP_CSR) {
        P->csr = *(const kl_csr_t *)op->user;
        P->op.user = &P->csr;
    }
    if (P->op.kind == KL_OP_STENCIL5) {
        const kl_stencil5_t *w = (const kl_stencil5_t *)op->user;
        if (!w) return c->fail(KL_ERR_INVALID, "KL_OP_STENCIL5 without weights");
        if (!(std::isfinite(w->c) && std::isfinite(w->wl) && std::isfinite(w->wr) && std::isfinite(w->wd) &&
              std::isfinite(w->wu)))
            return c->fail(KL_ERR_INVALID, "KL_OP_STENCIL5: the weights must be finite");
        if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "KL_OP_STENCIL5 is single-GPU in this release");
        P->w5 = *w;
        P->op.user = &P->w5;     // the kernels' coefficients (op_coef) come from this copy
        if ((P->pc.kind == KL_PC_CBPR2 || P->pc.kind == KL_PC_CHEB) && (w->wl * w->wr < 0.0 || w->wd * w->wu < 0.0))
            return c->fail(KL_ERR_UNSUPPORTED, "KL_OP_STENCIL5 with a complex spectrum (wl*wr < 0 or wd*wu < 0): "
                                               "the Chebyshev preconditioners need a real interval");
    }
    if (P->op.kind == KL_OP_ANISO5_VAR) {
        const kl_aniso_var_t *cf = (const kl_aniso_var_t *)P->op.user;
        if (!cf || !cf->kx || !cf->ky) return c->fail(KL_ERR_INVALID, "KL_OP_ANISO5_VAR without coefficient arrays");
        if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "variable-coefficient operators are single-GPU only");
        if (ny > 65535) return c->fail(KL_ERR_UNSUPPORTED, "KL_OP_ANISO5_VAR: ny <= 65535");
    }
    if (P->op.kind == KL_OP_USER && !P->op.fn) return c->fail(KL_ERR_INVALID, "KL_OP_USER without callback");
    if (P->op.kind == KL_OP_USER && c->nranks > 1)
        return c->fail(KL_ERR_UNSUPPORTED, "user operators are single-GPU only");
    if (P->op.kind != KL_OP_ANISO5) { P->op.eps_x = 1.0; P->op.eps_y = 1.0; }
    P->nparams = nparams < 8 ? nparams : 8;
    for (int i = 0; i < 8; ++i) P->params[i] = (params && i < P->nparams) ? params[i] : 0.0;
    if ((P->pc.kind == KL_PC_CBPR2 || P->pc.kind == KL_PC_CHEB) && P->nparams < 2)
        return c->fail(KL_ERR_INVALID, "Chebyshev preconditioners need params(1:2)");
    if (P->pc.kind == KL_PC_JACOBI_CHEB) {
        if (P->op.kind != KL_OP_ANISO5_VAR && P->op.kind != KL_OP_CSR)
            return c->fail(KL_ERR_UNSUPPORTED, "KL_PC_JACOBI_CHEB needs KL_OP_ANISO5_VAR or KL_OP_CSR; constant-diagonal "
                                               "operators use KL_PC_CHEB with the interval scaled by their diagonal");
        if (P->pc.degree < 0) return c->fail(KL_ERR_INVALID, "KL_PC_JACOBI_CHEB: degree >= 0");
        if (P->pc.degree >= 1) {
            if (P->nparams < 2) return c->fail(KL_ERR_INVALID, "KL_PC_JACOBI_CHEB of degree >= 1 needs params(1:2)");
            const double a = P->params[0], b = P->params[1];
            if (!(std::isfinite(a) && std::isfinite(b) && a > 0.0 && b > 0.0 && a != b))
                return c->fail(KL_ERR_INVALID, "KL_PC_JACOBI_CHEB: params(1:2) must be distinct finite positive numbers");
        }
    }
    P->nx = nx;
    P->ny = ny;
    kl_partition(c, ny, &P->j0, &P->nyl);
    if (P->nyl < 1) return c->fail(KL_ERR_INVALID, "more ranks than grid lines");
    P->n = (size_t)nx * P->nyl;
    KL_CUDA(c, cudaSetDevice(c->device));
    if (P->op.kind == KL_OP_CSR && validate) KL_TRY(csr_validate(c, &P->csr, nx, P->pc.kind == KL_PC_JACOBI_CHEB));
    if (c->nranks > 1) {
        size_t need = (size_t)nx * 8 * kChainMaxL;  // 4 slots x {lo,hi} x up to kChainMaxL lines (chained kernels)
        if (c->halo_doubles < need) {
            cudaStreamSynchronize(c->stream);
            cudaFree(c->d_halo);
            c->d_halo = nullptr;
            cudaError_t e = cudaMalloc(&c->d_halo, need * sizeof(double));
            if (e != cudaSuccess) return c->fail(KL_ERR_ALLOC, "halo buffers", e);
            c->halo_doubles = need;
        }
    }
    return KL_OK;
}

int halo_exchange(Prob *P, const double *const *vecs, int nvec, Halo *H) {
    Ctx *c = P->c;
    for (int a = 0; a < 4; ++a) H->lo[a] = H->hi[a] = nullptr;
    if (c->nranks == 1) return KL_OK;
    if (nvec > 4) return c->fail(KL_ERR_INVALID, "halo_exchange: too many vectors");
    const double *slo[4], *shi[4];
    for (int a = 0; a < nvec; ++a) {
        slo[a] = vecs[a];
        shi[a] = vecs[a] + (size_t)(P->nyl - 1) * P->nx;
    }
    // NOTE: a stencil kernel treats lo[0]==nullptr as "no lower neighbour" for all inputs.
    return comm_halo_exchange(c, slo, shi, H->lo, H->hi, nvec, P->nx);
}

// L-line halo for the temporally blocked kernels: lo = the lower neighbour's last `nlines` lines (grid lines
// -nlines..-1 in order), hi = the upper neighbour's first `nlines` lines.  Needs nyl >= nlines on every rank.
int halo_exchange_lines(Prob *P, const double *const *vecs, int nvec, int nlines, Halo *H) {
    Ctx *c = P->c;
    for (int a = 0; a < 4; ++a) H->lo[a] = H->hi[a] = nullptr;
    if (c->nranks == 1) return KL_OK;
    if (nvec > 4 || nlines < 1 || nlines > P->nyl) return c->fail(KL_ERR_INVALID, "halo_exchange_lines: bad arguments");
    const double *slo[4], *shi[4];
    for (int a = 0; a < nvec; ++a) {
        slo[a] = vecs[a];
        shi[a] = vecs[a] + (size_t)(P->nyl - nlines) * P->nx;
    }
    return comm_halo_exchange(c, slo, shi, H->lo, H->hi, nvec, nlines * P->nx);
}

// Variable-coefficient anisotropic diffusion, y = A(kx, ky) x (definition and evaluation order: oracle/krylov_extras.c
// ko_aniso_var).  One thread per pair of grid points, neighbours through L1/L2; the operator takes the generic solver
// path (one kernel per reference loop), like a user operator.  32n B (x, kx, ky in, y out).
__global__ void __launch_bounds__(256)
k_aniso_var(const double *__restrict__ x, double *__restrict__ y, const double *__restrict__ kx,
            const double *__restrict__ ky, const int nx, const int ny, const int *__restrict__ flags) {
    if (flags && flags[I_CONV_AT] >= 0) return;
    const int i = blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
    if (i >= nx) return;
    const size_t idx = (size_t)i + (size_t)j * nx;
    const double kxc = __ldg(kx + idx), kyc = __ldg(ky + idx), xc = __ldg(x + idx);
    const bool hl = i > 0, hr = i < nx - 1, hu = j > 0, hd = j < ny - 1;
    const double wl = hl ? 0.5 * (kxc + __ldg(kx + idx - 1)) : kxc, wr = hr ? 0.5 * (kxc + __ldg(kx + idx + 1)) : kxc;
    const double wu = hu ? 0.5 * (kyc + __ldg(ky + idx - nx)) : kyc, wd = hd ? 0.5 * (kyc + __ldg(ky + idx + nx)) : kyc;
    const double xl = hl ? __ldg(x + idx - 1) : 0.0, xr = hr ? __ldg(x + idx + 1) : 0.0;
    const double xd = hd ? __ldg(x + idx + nx) : 0.0, xu = hu ? __ldg(x + idx - nx) : 0.0;
    const double diag = ((wl + wr) + wd) + wu;
    const double s = fma(wl, xl, wr * xr), t = fma(wd, xd, wu * xu);
    y[idx] = fma(diag, xc, -(s + t));
}

// Jacobi-scaled Chebyshev on KL_OP_ANISO5_VAR, one pass per step (definition: tests/jacobi_cheb_twin.c;
// same arithmetic per point as the chained ChJacCheb, kl_chain_tma.cuh).  Serves odd nx, nx < 64, the chain switched
// off (KL_OPT_TMA / KL_OPT_FUSE / KL_OPT_CHAIN) and every step beyond kChainMaxL.  dinv = RN(1/diag) is recomputed
// from kx, ky in every pass.  kind 2: z = r*dinv (degree 0) ; kind 1: the start, d = z = (r*dinv)/theta ;
// kind 0: one step, d = fma(c1, d, c2*((r - A zin)*dinv)), z = zin + d.  Step: 56n B (r, zin, d, kx, ky in; d, z out).
__global__ void __launch_bounds__(256)
k_jacobi_cheb_step(const double *__restrict__ r, const double *__restrict__ zin, double *__restrict__ d,
                   double *__restrict__ z, const double *__restrict__ kx, const double *__restrict__ ky, const int nx,
                   const int ny, const double theta, const double c1, const double c2, const int kind,
                   const int *__restrict__ flags) {
    if (flags && flags[I_CONV_AT] >= 0) return;
    const int i = blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
    if (i >= nx) return;
    const size_t idx = (size_t)i + (size_t)j * nx;
    const double kxc = __ldg(kx + idx), kyc = __ldg(ky + idx);
    const bool hl = i > 0, hr = i < nx - 1, hu = j > 0, hd = j < ny - 1;
    const double wl = hl ? 0.5 * (kxc + __ldg(kx + idx - 1)) : kxc, wr = hr ? 0.5 * (kxc + __ldg(kx + idx + 1)) : kxc;
    const double wu = hu ? 0.5 * (kyc + __ldg(ky + idx - nx)) : kyc, wd = hd ? 0.5 * (kyc + __ldg(ky + idx + nx)) : kyc;
    const double diag = ((wl + wr) + wd) + wu;
    const double dinv = __drcp_rn(diag), rc = __ldg(r + idx);
    if (kind == 2) {
        z[idx] = rc * dinv;
        return;
    }
    if (kind == 1) {
        const double d0 = (rc * dinv) / theta;
        d[idx] = d0;
        z[idx] = d0;
        return;
    }
    const double xc = __ldg(zin + idx);
    const double xl = hl ? __ldg(zin + idx - 1) : 0.0, xr = hr ? __ldg(zin + idx + 1) : 0.0;
    const double xd = hd ? __ldg(zin + idx + nx) : 0.0, xu = hu ? __ldg(zin + idx - nx) : 0.0;
    const double s = fma(wl, xl, wr * xr), t = fma(wd, xd, wu * xu);
    const double az = fma(diag, xc, -(s + t));
    const double dn = fma(c1, d[idx], c2 * ((rc - az) * dinv));
    d[idx] = dn;
    z[idx] = xc + dn;
}

int op_apply(Prob *P, const double *x, double *y, bool gated) {
    Ctx *c = P->c;
    if (P->op.kind == KL_OP_ANISO5_VAR) {
        const kl_aniso_var_t *cf = (const kl_aniso_var_t *)P->op.user;
        dim3 grid((unsigned)((P->nx + 255) / 256), (unsigned)P->nyl);
        k_aniso_var<<<grid, 256, 0, c->stream>>>(x, y, cf->kx, cf->ky, P->nx, P->nyl, gated ? c->d_I : nullptr);
        c->stats.kernel_launches++;
        return KL_OK;
    }
    if (P->op.kind == KL_OP_DENSE) return launch_gemv(c, (const double *)P->op.user, P->nx, x, y, gated);
    if (P->op.kind == KL_OP_CSR) return launch_csr_spmv(c, &P->csr, P->nx, x, y, gated);
    if (!P->builtin_op()) {
        // user callbacks cannot be gated on the device flag; they run unconditionally
        int rc = P->op.fn(P->op.user, x, y, P->nx, P->nyl, (void *)c->stream);
        if (rc != 0) return c->fail(KL_ERR_INVALID, "user operator failed");
        return KL_OK;
    }
    Halo H;
    const double *vecs[1] = {x};
    KL_TRY(halo_exchange(P, vecs, 1, &H));
    FApply f;
    set_io(f, P, vecs, H);
    set_gate(f, c, gated);
    f.y = y;
    return launch_stencil(c, &P->op, f, P->nx, P->nyl, NoPost{});
}

int op_resid(Prob *P, const double *x, const double *b, double *z, bool gated) {
    Ctx *c = P->c;
    if (!P->builtin_op()) {
        KL_TRY(op_apply(P, x, z, gated));
        double one = 1.0;
        KL_CUDA(c, cudaMemcpyAsync(c->d_S + S_TMP3, &one, sizeof(double), cudaMemcpyHostToDevice, c->stream));
        PAxpy t;
        set_gate(t, c, gated);
        t.a = b; t.b = z; t.y = z; t.S = c->d_S; t.s_idx = S_TMP3; t.sign = -1.0;
        return launch_pointwise(c, t, P->n, NoPost{});
    }
    Halo H;
    const double *vecs[1] = {x};
    KL_TRY(halo_exchange(P, vecs, 1, &H));
    FResid f;
    set_io(f, P, vecs, H);
    set_gate(f, c, gated);
    f.b = b;
    f.z = z;
    return launch_stencil(c, &P->op, f, P->nx, P->nyl, NoPost{});
}

// Chebyshev degree-k step (see oracle/krylov_extras.c ko_cheb):
//   first: u = r/theta (= d_old) ; else u = z_old (in[0]), d_old from memory
//   d_new = fma(c1, d_old, c2*(r - A u)) ; z_new = u + d_new
template <int MODE>
struct FChebStep : StencilBase<1, (MODE ? 1 : 0)> {
    const double *r;
    double *d, *z_new;
    double theta, c1, c2;
    int first;
    FastDiv fd;
    __device__ __forceinline__ void init() { fd.set(theta); }
    __device__ __forceinline__ double point(const double (&v)[1]) const { return first ? fd.div(v[0]) : v[0]; }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[1][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
        double rr[VEC], dd[VEC], zz[VEC];
        if (first) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) { rr[v] = raw[0][v]; dd[v] = cu[v]; }
        } else {
            KL_LD(VEC, rr, r, idx)
            if (VEC == 2) {
                double2 t = *reinterpret_cast<const double2 *>(d + idx);
                dd[0] = t.x; dd[VEC - 1] = t.y;
            } else {
                dd[0] = d[idx];
            }
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            dd[v] = fma(c1, dd[v], c2 * (rr[v] - au[v]));
            zz[v] = cu[v] + dd[v];
            if (MODE == 1) acc[0] = fma(zz[v], zz[v], acc[0]);
            if (MODE == 2) acc[0] = fma(rr[v], zz[v], acc[0]);
        }
        KL_ST(VEC, d, idx, dd)
        KL_ST(VEC, z_new, idx, zz)
    }
};

// KL_PC_JACOBI_CHEB (prob_init admits it on KL_OP_ANISO5_VAR and KL_OP_CSR only, which run on one GPU)
static int pc_jacobi_cheb(Prob *P, const double *r, double *z, double *aux, double *aux2, int mode, bool gated,
                          const PostAny &post) {
    Ctx *c = P->c;
    const bool csr = P->op.kind == KL_OP_CSR;
    const kl_aniso_var_t *cf = (const kl_aniso_var_t *)P->op.user;   // KL_OP_ANISO5_VAR only
    const int k = P->pc.degree;
    const dim3 grid((unsigned)((P->nx + 255) / 256), (unsigned)P->nyl);
    const int *flags = gated ? c->d_I : nullptr;
    auto pass = [&](const double *zin, double *zout, double theta, double c1, double c2, int kind) {
        if (csr) {
            launch_csr_jacobi_cheb_step(c, &P->csr, P->nx, r, zin, aux2, zout, theta, c1, c2, kind, gated);
            return;
        }
        k_jacobi_cheb_step<<<grid, 256, 0, c->stream>>>(r, zin, aux2, zout, cf->kx, cf->ky, P->nx, P->nyl, theta, c1, c2,
                                                        kind, flags);
        c->stats.kernel_launches++;
    };
    if (k == 0) {
        pass(nullptr, z, 0.0, 0.0, 0.0, 2);
    } else {
        // Saad Alg. 12.1 on D^-1 A; coefficients on the host (same arithmetic as the oracle and KL_PC_CHEB)
        const double ea = P->params[0], eb = P->params[1];
        const double theta = (eb + ea) / 2.0, delta = fabs(eb - ea) / 2.0;
        const double sigma = theta / delta;
        double rho_prev = 1.0 / sigma;
        // ping-pong so that the final result lands in z: z_s lives in zb[(k - s) & 1], d in aux2
        double *zb[2] = {z, aux};
        const int kc = k < kChainMaxL ? k : kChainMaxL;
        int s0 = 0;
        // chain_ok looks at the grid only; the chained ChJacCheb reads the aniso_var coefficient fields
        if (!csr && chain_ok(P, kc)) {
            // the first min(k, 6) steps in ONE pass over r, kx, ky (kl_chain_tma.cuh ChJacCheb): 32n B
            double c1s[kChainMaxL], c2s[kChainMaxL];
            for (int s = 0; s < kc; ++s) {
                const double rho = 1.0 / (2.0 * sigma - rho_prev);
                c1s[s] = rho * rho_prev;
                c2s[s] = 2.0 * rho / delta;
                rho_prev = rho;
            }
            const double *in[3] = {r, cf->kx, cf->ky};
            const Halo H = {};
            double *dst = (kc == k) ? z : zb[(k - kc) & 1];
#define KL_JC(LL)                                                                       \
    case LL: {                                                                          \
        ChJacCheb<LL> f;                                                                \
        set_io(f, P, in, H);                                                            \
        set_gate(f, c, gated);                                                          \
        f.z = dst; f.d_out = (kc == k) ? nullptr : aux2; f.mode = (kc == k) ? mode : 0; \
        f.theta = theta;                                                                \
        for (int s = 0; s < LL; ++s) { f.c1[s] = c1s[s]; f.c2[s] = c2s[s]; }            \
        if (kc == k && mode != 0) { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, post, mode == 2 ? 1 : 0)); } \
        else { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, NoPost{})); }           \
    } break;
            switch (kc) {
                KL_JC(1) KL_JC(2) KL_JC(3) KL_JC(4) KL_JC(5) KL_JC(6)
                default: return c->fail(KL_ERR_INVALID, "jacobi-chebyshev chain length");
            }
#undef KL_JC
            if (kc == k) return KL_OK;
            s0 = kc;
        } else {
            pass(nullptr, zb[k & 1], theta, 0.0, 0.0, 1);
        }
        for (int s = s0; s < k; ++s) {
            const double rho = 1.0 / (2.0 * sigma - rho_prev);
            pass(zb[(k - s) & 1], zb[(k - s - 1) & 1], theta, rho * rho_prev, 2.0 * rho / delta, 0);
            rho_prev = rho;
        }
    }
    if (mode != 0) {
        PDot2 dt;
        set_gate(dt, c, gated);
        dt.a = (mode == 1) ? z : r; dt.b = z; dt.c = nullptr; dt.d = nullptr;
        KL_TRY(launch_pointwise(c, dt, P->n, post));
    }
    return KL_OK;
}

int pc_apply_any(Prob *P, const double *r, double *z, double *aux, double *aux2, int mode, bool gated,
                 const PostAny &post) {
    Ctx *c = P->c;
    const int kind = P->pc.kind;
    if (kind == KL_PC_JACOBI_CHEB) return pc_jacobi_cheb(P, r, z, aux, aux2, mode, gated, post);
    if (kind == KL_PC_CBPR2 && P->builtin_op()) {
        Cbpr2Coef cf = cbpr2_coef(P->params);
        Halo H;
        const double *vecs[1] = {r};
        KL_TRY(halo_exchange(P, vecs, 1, &H));
#define KL_CB(MODE)                                     \
    {                                                   \
        FCbpr2<MODE> f;                                 \
        set_io(f, P, vecs, H);                          \
        set_gate(f, c, gated);                          \
        f.z = z;                                        \
        f.d = cf.d;                                     \
        f.alpha = cf.alpha;                             \
        return launch_stencil(c, &P->op, f, P->nx, P->nyl, post); \
    }
        if (mode == 0) KL_CB(0) else if (mode == 1) KL_CB(1) else KL_CB(2)
#undef KL_CB
    }
    if (kind == KL_PC_CHEB && P->builtin_op() && P->pc.degree >= 1) {
        // Saad Alg. 12.1; coefficients on the host (same arithmetic as the oracle)
        double ea = P->params[0], eb = P->params[1];
        double theta = (eb + ea) / 2.0, delta = fabs(eb - ea) / 2.0;
        double sigma = theta / delta, rho_prev = 1.0 / sigma;
        const int k = P->pc.degree;
        int s0 = 0;
        // ping-pong so that the final result lands in z: z_k = z if k odd else aux
        double *zb[2] = {z, aux};
        // degree <= 6: one chain ; 7..12: two balanced chains (the second continues from the stored z and d) ;
        // above: a chain of 6 and one pass per remaining step
        const bool two = k > kChainMaxL && k <= 2 * kChainMaxL;
        const int kc = two ? (k + 1) / 2 : (k < kChainMaxL ? k : kChainMaxL);
        if (chain_ok(P, kc)) {
            // the first min(k, 6) steps in ONE pass over r (kl_chain_tma.cuh): 16n B instead of 40n B per step
            Halo H;
            const double *hv[1] = {r};
            KL_TRY(halo_exchange_lines(P, hv, 1, kc, &H));
            double c1s[kChainMaxL], c2s[kChainMaxL];
            for (int s = 0; s < kc; ++s) {
                double rho = 1.0 / (2.0 * sigma - rho_prev);
                c1s[s] = rho * rho_prev;
                c2s[s] = 2.0 * rho / delta;
                rho_prev = rho;
            }
            double *dst = (kc == k) ? z : (two ? aux : zb[(k - kc) & 1]);
#define KL_CC(LL)                                                                       \
    case LL: {                                                                          \
        ChCheb<LL> f;                                                                   \
        set_io(f, P, hv, H);                                                            \
        set_gate(f, c, gated);                                                          \
        f.z = dst; f.d_out = (kc == k) ? nullptr : aux2; f.mode = (kc == k) ? mode : 0; \
        f.theta = theta;                                                                \
        for (int s = 0; s < LL; ++s) { f.c1[s] = c1s[s]; f.c2[s] = c2s[s]; }            \
        if (kc == k && mode != 0) { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, post, mode == 2 ? 1 : 0)); } \
        else { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, NoPost{})); }           \
    } break;
            switch (kc) {
                KL_CC(1) KL_CC(2) KL_CC(3) KL_CC(4) KL_CC(5) KL_CC(6)
                default: return c->fail(KL_ERR_INVALID, "chebyshev chain length");
            }
#undef KL_CC
            if (kc == k) return KL_OK;
            if (two) {
                // second chain: (z_kc, d_kc, r) -> z_k.  Inputs aux, aux2 ; output z.
                const int kb = k - kc;
                Halo H2;
                const double *hv3[3] = {aux, aux2, r};
                KL_TRY(halo_exchange_lines(P, hv3, 3, kb, &H2));
                for (int s = 0; s < kb; ++s) {
                    double rho = 1.0 / (2.0 * sigma - rho_prev);
                    c1s[s] = rho * rho_prev;
                    c2s[s] = 2.0 * rho / delta;
                    rho_prev = rho;
                }
#define KL_CT(LL)                                                                       \
    case LL: {                                                                          \
        ChChebCont<LL> f;                                                               \
        set_io(f, P, hv3, H2);                                                          \
        set_gate(f, c, gated);                                                          \
        f.z = z; f.mode = mode;                                                         \
        for (int s = 0; s < LL; ++s) { f.c1[s] = c1s[s]; f.c2[s] = c2s[s]; }            \
        if (mode != 0) { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, post, mode == 2 ? 1 : 0)); } \
        else { KL_TRY(launch_chain(c, &P->op, f, P->nx, P->nyl, NoPost{})); }           \
    } break;
                switch (kb) {
                    KL_CT(3) KL_CT(4) KL_CT(5) KL_CT(6)      // kb = k - ceil(k/2) for k = 7..12
                    default: return c->fail(KL_ERR_INVALID, "chebyshev chain length");
                }
#undef KL_CT
                return KL_OK;
            }
            s0 = kc;
        }
        for (int s = s0; s < k; ++s) {
            double rho = 1.0 / (2.0 * sigma - rho_prev);
            double c1 = rho * rho_prev, c2 = 2.0 * rho / delta;
            const double *src = (s == 0) ? r : zb[(k - s) & 1];
            double *dst = zb[(k - s - 1) & 1];
            Halo H;
            const double *vecs[1] = {src};
            KL_TRY(halo_exchange(P, vecs, 1, &H));
            const int m = (s == k - 1) ? mode : 0;
#define KL_CH(MODE)                                                       \
    {                                                                     \
        FChebStep<MODE> f;                                                \
        set_io(f, P, vecs, H);                                            \
        set_gate(f, c, gated);                                            \
        f.r = r; f.d = aux2; f.z_new = dst;                               \
        f.theta = theta; f.c1 = c1; f.c2 = c2; f.first = (s == 0);        \
        if (MODE == 0) { KL_TRY(launch_stencil(c, &P->op, f, P->nx, P->nyl, NoPost{})); } \
        else { KL_TRY(launch_stencil(c, &P->op, f, P->nx, P->nyl, post)); } \
    }
            if (m == 0) KL_CH(0) else if (m == 1) KL_CH(1) else KL_CH(2)
#undef KL_CH
            rho_prev = rho;
        }
        return KL_OK;
    }
    // generic path: KL_PC_NONE, user preconditioner, or built-in preconditioner on a user operator
    if (kind == KL_PC_NONE) {
        if (z != r) {
            // gated copy
            PCopy f;
            set_gate(f, c, gated);
            f.a = r; f.y = z;
            KL_TRY(launch_pointwise(c, f, P->n, NoPost{}));
        }
    } else if (kind == KL_PC_USER) {
        if (!P->pc.fn) return c->fail(KL_ERR_INVALID, "KL_PC_USER without callback");
        int rc = P->pc.fn(c, &P->op, P->pc.user, r, z, aux, P->params, P->nparams, P->nx, P->nyl,
                          (void *)c->stream);
        if (rc != 0) return c->fail(KL_ERR_INVALID, "user preconditioner failed");
    } else if (kind == KL_PC_CBPR2) {
        // user operator: the reference's three loops (chebyshev.f90:27-37)
        Cbpr2Coef cf = cbpr2_coef(P->params);
        cudaMemcpyAsync(c->d_S + S_CD, &cf.d, sizeof(double), cudaMemcpyHostToDevice, c->stream);
        PScale s;
        set_gate(s, c, gated);
        s.in = r; s.out = z; s.S = c->d_S; s.s_idx = S_CD;
        KL_TRY(launch_pointwise(c, s, P->n, NoPost{}));
        KL_TRY(op_apply(P, z, aux, gated));
        // z = z + alpha*(r - aux): t = r - aux (in aux), then z += alpha*t
        cudaMemcpyAsync(c->d_S + S_CALPHA, &cf.alpha, sizeof(double), cudaMemcpyHostToDevice, c->stream);
        double one = 1.0;
        cudaMemcpyAsync(c->d_S + S_TMP3, &one, sizeof(double), cudaMemcpyHostToDevice, c->stream);
        PAxpy t;
        set_gate(t, c, gated);
        t.a = r; t.b = aux; t.y = aux; t.S = c->d_S; t.s_idx = S_TMP3; t.sign = -1.0;
        KL_TRY(launch_pointwise(c, t, P->n, NoPost{}));
        PAxpy u;
        set_gate(u, c, gated);
        u.a = z; u.b = aux; u.y = z; u.S = c->d_S; u.s_idx = S_CALPHA; u.sign = 1.0;
        KL_TRY(launch_pointwise(c, u, P->n, NoPost{}));
    } else {
        return c->fail(KL_ERR_UNSUPPORTED, "preconditioner kind not supported with this operator");
    }
    if (mode != 0) {
        PDot2 dt;
        set_gate(dt, c, gated);
        dt.a = (mode == 1) ? z : r; dt.b = z; dt.c = nullptr; dt.d = nullptr;
        // PDot2 has NRED = 2; post reads S_RED[0] only
        KL_TRY(launch_pointwise(c, dt, P->n, post));
    }
    return KL_OK;
}


int stage_in(Ctx *c, double *d_dst, const double *src, size_t n) {
    cudaMemcpyKind k = c->pointer_mode == KL_POINTER_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    if (c->pointer_mode == KL_POINTER_DEVICE && d_dst == src) return KL_OK;
    KL_CUDA(c, cudaMemcpyAsync(d_dst, src, n * sizeof(double), k, c->stream));
    if (k == cudaMemcpyHostToDevice) c->stats.h2d_bytes += (double)n * sizeof(double);
    return KL_OK;
}
int stage_out(Ctx *c, double *dst, const double *d_src, size_t n) {
    cudaMemcpyKind k = c->pointer_mode == KL_POINTER_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    if (c->pointer_mode == KL_POINTER_DEVICE && dst == d_src) return KL_OK;
    KL_CUDA(c, cudaMemcpyAsync(dst, d_src, n * sizeof(double), k, c->stream));
    if (k == cudaMemcpyDeviceToHost) c->stats.d2h_bytes += (double)n * sizeof(double);
    return KL_OK;
}

int read_back(Ctx *c) {
    KL_CUDA(c, cudaMemcpyAsync(c->h_pinned, c->d_S, sizeof(double) * 64, cudaMemcpyDeviceToHost, c->stream));
    KL_CUDA(c, cudaMemcpyAsync(c->h_pinned_i, c->d_I, sizeof(int) * I_COUNT, cudaMemcpyDeviceToHost, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    return KL_OK;
}

int x0_check(Ctx *c, const double *b, const double *x) {
    if (!c->opt_x0) return KL_OK;
    // multi-GPU: the plain-CG producer-push prologue pushes r0's boundary lines, a path that is not covered yet
    if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "KL_OPT_X0 is single-GPU in this release");
    if (c->pointer_mode == KL_POINTER_DEVICE && x == b)
        return c->fail(KL_ERR_INVALID, "KL_OPT_X0: x is read as the initial guess and written as the solution, it must not be b");
    return KL_OK;
}

int x0_norm(Ctx *c, const double *v, size_t n, double *norm) {
    PDot2 d;
    set_gate(d, c, false);
    d.a = v; d.b = v; d.c = nullptr; d.d = nullptr;
    KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_RES, 1}));
    KL_TRY(read_back(c));
    *norm = c->h_pinned[S_RES];
    KL_CUDA(c, cudaMemsetAsync(c->d_S + S_RES, 0, sizeof(double), c->stream));
    return KL_OK;
}

int x0_zero_step(Ctx *c) {
    c->history.clear();
    c->history_len = 0;
    KL_CUDA(c, cudaEventRecord(c->ev3, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev2, c->ev3);
    c->stats.total_ms = ms;
    return KL_OK;
}

int fetch_history(Ctx *c) {
    KL_TRY(read_back(c));
    int len = c->h_pinned_i[I_HIST];
    c->history_len = len;
    int k = len < c->hist_cap ? len : c->hist_cap;
    c->history.resize(k);
    if (k > 0) {
        KL_CUDA(c, cudaMemcpyAsync(c->history.data(), c->d_hist, sizeof(double) * k, cudaMemcpyDeviceToHost, c->stream));
        KL_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return KL_OK;
}

}  // namespace kl

using namespace kl;

extern "C" {

// The operator is the Kronecker sum of two tridiagonal Toeplitz matrices, tridiag(-wl, c/2, -wr) (x) I + I (x)
// tridiag(-wu, c/2, -wd).  With wl*wr >= 0 and wd*wu >= 0 each factor is diagonally similar to a symmetric one, with
// eigenvalues c/2 - 2 sqrt(wl*wr) cos(k pi/(nx+1)), k = 1..nx (and the same in y); the extremes are k = 1 and k = nx.
int kl_stencil5_spectrum(const kl_stencil5_t *w, int nx, int ny, double *lam_min, double *lam_max) {
    if (!w || !lam_min || !lam_max) return KL_ERR_INVALID;
    *lam_min = *lam_max = NAN;
    if (nx < 1 || ny < 1) return KL_ERR_INVALID;
    if (!(std::isfinite(w->c) && std::isfinite(w->wl) && std::isfinite(w->wr) && std::isfinite(w->wd) &&
          std::isfinite(w->wu)))
        return KL_ERR_INVALID;
    const double gx = w->wl * w->wr, gy = w->wd * w->wu;
    if (gx < 0.0 || gy < 0.0) return KL_ERR_UNSUPPORTED;
    const double pi = 3.14159265358979323846;
    const double ax = 2.0 * std::sqrt(gx) * std::cos(pi / (nx + 1)), ay = 2.0 * std::sqrt(gy) * std::cos(pi / (ny + 1));
    *lam_min = (w->c - ax) - ay;
    *lam_max = (w->c + ax) + ay;
    return KL_OK;
}

int kl_apply_operator(kl_handle_t h, const kl_operator_t *A_x, const double *x, double *y, int nx, int ny) {
    if (!h || !A_x || !x || !y) return KL_ERR_INVALID;
    Ctx *c = h;
    Prob P;
    // device pointer mode stays enqueue-only (it may run inside a KL_PC_USER callback): no KL_OP_CSR check
    KL_TRY(prob_init(&P, c, A_x, nullptr, nullptr, 0, nx, ny, c->pointer_mode != KL_POINTER_DEVICE));
    if (c->pointer_mode == KL_POINTER_DEVICE) {
        KL_TRY(op_apply(&P, x, y, false));
        return KL_OK;
    }
    KL_TRY(ws_reserve(c, 2 * ws_need(P.n)));
    ws_reset(c);
    double *dx = ws_take<double>(c, P.n), *dy = ws_take<double>(c, P.n);
    KL_TRY(stage_in(c, dx, x, P.n));
    KL_TRY(op_apply(&P, dx, dy, false));
    KL_TRY(stage_out(c, y, dy, P.n));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    return KL_OK;
}

int kl_apply_precond(kl_handle_t h, const kl_precond_t *M_inv, const kl_operator_t *A_x, const double *r,
                     double *z, const double *params, int nparams, int nx, int ny) {
    if (!h || !A_x || !M_inv || !r || !z) return KL_ERR_INVALID;
    Ctx *c = h;
    Prob P;
    KL_TRY(prob_init(&P, c, A_x, M_inv, params, nparams, nx, ny, c->pointer_mode != KL_POINTER_DEVICE));
    KL_TRY(ws_reserve(c, 4 * ws_need(P.n)));
    ws_reset(c);
    if (c->pointer_mode == KL_POINTER_DEVICE && r != z) {
        // device vectors are used in place (stream-ordered, returns after enqueue like kl_apply_operator)
        double *aux = ws_take<double>(c, P.n), *aux2 = ws_take<double>(c, P.n);
        KL_TRY(pc_apply(&P, r, z, aux, aux2, 0, false, NoPost{}));
        KL_CUDA(c, cudaGetLastError());
        return KL_OK;
    }
    double *dr = ws_take<double>(c, P.n), *dz = ws_take<double>(c, P.n);
    double *aux = ws_take<double>(c, P.n), *aux2 = ws_take<double>(c, P.n);
    KL_TRY(stage_in(c, dr, r, P.n));
    KL_TRY(pc_apply(&P, dr, dz, aux, aux2, 0, false, NoPost{}));
    KL_TRY(stage_out(c, z, dz, P.n));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    return KL_OK;
}

}  // extern "C"
