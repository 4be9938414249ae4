// kl_ops.cuh -- problem descriptor, halo exchange, operator / preconditioner application.
#pragma once
#include "kl_functors.cuh"
#include "kl_chain_tma.cuh"

namespace kl {

struct Prob {
    Ctx *c;
    kl_operator_t op;
    kl_precond_t pc;
    double params[8];
    int nparams;
    int nx, ny;        // global grid
    int nyl, j0;       // this rank's slab
    size_t n;          // nx * nyl
    // KL_OP_STENCIL5: the caller's weights, copied at the start of the call (op.user points here); all zero for the
    // other kinds.  Part of every CUDA-graph key.
    kl_stencil5_t w5;
    bool builtin_op() const {   // the stencil operators (fused kernels); user callbacks and dense matrices take the generic path
        return op.kind == KL_OP_POISSON5 || op.kind == KL_OP_POISSON5_BRANCHY || op.kind == KL_OP_ANISO5 ||
               op.kind == KL_OP_STENCIL5;
    }
    // false only for a KL_OP_STENCIL5 that is not symmetric (CG, PCG and Lanczos refuse it)
    bool symmetric() const { return op.kind != KL_OP_STENCIL5 || (w5.wl == w5.wr && w5.wd == w5.wu); }
};

int prob_init(Prob *P, Ctx *c, const kl_operator_t *op, const kl_precond_t *pc, const double *params,
              int nparams, int nx, int ny);

// Halo buffers: slot s in [0,4) -> lo/hi line of nx doubles each.
struct Halo {
    const double *lo[4];
    const double *hi[4];
};
// exchange the boundary lines of `nvec` vectors; fills H (nullptr at the global
// boundary / single GPU).
int halo_exchange(Prob *P, const double *const *vecs, int nvec, Halo *H);

int halo_exchange_lines(Prob *P, const double *const *vecs, int nvec, int nlines, Halo *H);
// can the temporally blocked kernels run L levels on this problem?  (all ranks take the same decision)
inline bool chain_ok(const Prob *P, int L) {
    const Ctx *c = P->c;
    if (!(c->opt_tma && c->opt_fuse && c->opt_chain) || P->nx % 2 != 0 || P->nx < 64) return false;
    // stv_poisson (the reference's branchy variant, unused by its drivers) runs one pass per application: the
    // temporally blocked kernels are only instantiated for stvec and the constant-coefficient operators
    // (KL_OP_ANISO5, and KL_OP_STENCIL5 on one GPU)
    if (P->op.kind == KL_OP_POISSON5_BRANCHY) return false;
    if (c->nranks == 1) return true;
    return P->ny / c->nranks >= L && (size_t)L * P->nx <= 65536;   // L-line halo fits the exchange buffers
}

template <class F>
inline void set_io(F &f, const Prob *P, const double *const *vecs, const Halo &H) {
    for (int a = 0; a < F::NIN; ++a) {
        f.in[a] = vecs[a];
        f.lo[a] = H.lo[a];
        f.hi[a] = H.hi[a];
    }
}
template <class F>
inline void set_gate(F &f, const Ctx *c, bool gated, int step = 0, int run_on_conv = 0) {
    f.flags = gated ? c->d_I : nullptr;
    f.step = step;
    f.run_on_conv = run_on_conv;
}

// y = A x
int op_apply(Prob *P, const double *x, double *y, bool gated);
// y = matmul(A, x) for a dense column-major n x n matrix in device memory (kl_dense.cu)
int launch_gemv(Ctx *c, const double *dA, int n, const double *x, double *y, bool gated);
// solver bodies shared by the stencil and the dense entry points
int gmres_mgsr_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny, int m, double tol,
                     double *final_err, double *v_err, int *n_out_p, int *restart_out_p, const kl_precond_t *M,
                     const double *params, int nparams, int mf);
int gmres_hh_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny, int m, double tol,
                   double *final_err, double *v_err, int *n_out_p, int *stages_out_p, const kl_precond_t *M,
                   const double *params, int nparams, int prec_variant);
// z = b - A x
int op_resid(Prob *P, const double *x, const double *b, double *z, bool gated);
// z = M^-1 r ; mode 0: no reduction, 1: S_RED[0] = sum z*z, 2: S_RED[0] = sum r*z.
// aux/aux2: scratch vectors (aux2 only needed for KL_PC_CHEB and KL_PC_JACOBI_CHEB).  For KL_PC_NONE
// z = r is a copy.  `post` runs after the reduction (mode != 0).
// (compiled once, in kl_ops.cu: the post functor is a run-time PostAny, so the Chebyshev chain kernels and the
// cbpr2 / Chebyshev-step stencil kernels are instantiated in ONE translation unit instead of in every solver's)
int pc_apply_any(Prob *P, const double *r, double *z, double *aux, double *aux2, int mode, bool gated,
                 const PostAny &post);
template <class Post>
inline int pc_apply(Prob *P, const double *r, double *z, double *aux, double *aux2, int mode, bool gated,
                    const Post &post) {
    return pc_apply_any(P, r, z, aux, aux2, mode, gated, to_any(post));
}

// staging of user vectors according to the pointer mode
int stage_in(Ctx *c, double *d_dst, const double *src, size_t n);
int stage_out(Ctx *c, double *dst, const double *d_src, size_t n);

// read the scalar / int blocks back (async copy + sync)
int read_back(Ctx *c);
// copy history from the device and fill ctx->history
int fetch_history(Ctx *c);

// KL_OPT_X0 (x is the initial guess).  x0_check: the option's preconditions (one GPU; device mode: x is not b).
int x0_check(Ctx *c, const double *b, const double *x);
// ||v||, read back to the host, for the zero-step test before the first iteration.  S_RES, where the reduction
// lands, is zeroed again, so the iteration starts from the scalar block of a cold solve.
int x0_norm(Ctx *c, const double *v, size_t n, double *norm);
// bookkeeping of a zero-step return (x0 already meets the stopping test): empty history, call time
int x0_zero_step(Ctx *c);


}  // namespace kl
