/*
 * krylov_b200.h -- C ABI of libkrylov_b200.so, the B200 (sm_100a) implementation
 * of Krylov Lab's iterative-solver hot path.
 *
 * This header is the drop-in boundary: every entry point replaces one public
 * module procedure of the reference (AlexanderGSC/gmres, Fortran 2008) and keeps
 * its argument order and meaning.  The citation after each declaration is the
 * reference interface it replaces (path:line relative to the reference root).
 * The ISO_C_BINDING shim that gives the reference's Fortran drivers the original
 * procedure names on top of this ABI is fortran/krylov_b200.f90; the C++ mirror
 * is include/krylov_b200.hpp; INTEGRATION.md shows the bindings.
 *
 * Conventions
 *   - All arithmetic is IEEE FP64.  Grids are column-major with i fastest,
 *     idx = i + j*nx (0-based), exactly the reference's idx = i+(j-1)*n layout.
 *   - nx, ny are the GLOBAL grid extents.  With a multi-GPU communicator the
 *     grid is row-slab decomposed in memory order: rank p owns the contiguous
 *     lines j in [j0, j0+ny_local) (kl_partition) and every vector argument is
 *     that rank's local slab of nx*ny_local doubles.
 *   - b / x / vector arguments are HOST pointers by default, or DEVICE pointers
 *     after kl_set_pointer_mode(h, KL_POINTER_DEVICE) (vectors and the Krylov
 *     basis then stay resident in HBM between calls).  Small outputs
 *     (final_err, v_err, counters, res) are always host pointers.
 *   - Every function returns an int status (the reference has no error
 *     convention at all: failure there is NaN propagation or silently hitting
 *     the restart cap).  Outputs are always defined.
 *   - Calls are stream-ordered on the handle's stream; solver entry points
 *     block until the convergence information is on the host.  A handle is not
 *     thread-safe; distinct handles are independent.
 */
#ifndef KRYLOV_B200_H
#define KRYLOV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KL_VERSION 101

typedef struct kl_context_s *kl_handle_t;

/* ---- status codes ------------------------------------------------------ */
enum {
    KL_OK = 0,
    KL_NOT_CONVERGED = 1,   /* restart / iteration cap reached               */
    KL_BREAKDOWN = 2,       /* NaN / Inf or zero pivot met                   */
    KL_ERR_INVALID = -1,
    KL_ERR_CUDA = -2,
    KL_ERR_NCCL = -3,
    KL_ERR_ALLOC = -4,
    KL_ERR_UNSUPPORTED = -5
};

/* ---- operator plug-in: replaces procedure(stencil_vector) ---------------
 * src/interfaces.f90:12-18   subroutine stencil_vector(x, y, n)            */
typedef int (*kl_apply_fn)(void *user, const double *d_x, double *d_y, int nx, int ny_local,
                           void *cuda_stream); /* enqueue-only, must not synchronise */
enum {
    KL_OP_POISSON5 = 0,          /* poisson::stvec        src/problems/poisson.f90:33-77 */
    KL_OP_POISSON5_BRANCHY = 1,  /* poisson::stv_poisson  src/problems/poisson.f90:79-96 */
    KL_OP_ANISO5 = 2,            /* constant-coefficient anisotropic diffusion (README.md:46, new) */
    KL_OP_DENSE = 3,             /* dense column-major n x n matrix in device memory (`user`), nx = n, ny = 1;
                                    set up by kl_gmres_mgsr_dense / kl_gmres_hh_dense (single GPU only)   */
    KL_OP_ANISO5_VAR = 4,        /* variable-coefficient anisotropic diffusion, self-adjoint finite-volume form
                                    (README.md:46 WIP, new): `user` points to a kl_aniso_var_t (single GPU only) */
    KL_OP_STENCIL5 = 5,          /* general constant-coefficient 5-point operator, e.g. convection-diffusion (new):
                                    `user` points to a HOST kl_stencil5_t, read at the start of each call (single GPU
                                    only).  Nonsymmetric unless wl == wr and wd == wu: CG, PCG and kl_lanczos refuse it
                                    then (KL_ERR_UNSUPPORTED), and KL_PC_CBPR2 / KL_PC_CHEB refuse it when its spectrum
                                    is complex (wl*wr < 0 or wd*wu < 0).  It runs through the same fused and temporally
                                    blocked kernels as KL_OP_ANISO5.                                                 */
    KL_OP_USER = 100             /* user callback on device pointers (single GPU only) */
};
/* coefficient fields of KL_OP_ANISO5_VAR: cell values kx(i,j), ky(i,j), idx = i + j*nx, DEVICE pointers (kl_vec_alloc /
 * kl_vec_upload) that stay valid for the duration of the call.  A face carries the mean of its two cells.     */
typedef struct {
    const double *kx, *ky;
} kl_aniso_var_t;
/* weights of KL_OP_STENCIL5, finite numbers (idx = i + j*nx, "d" = idx+nx is line j+1, "u" = idx-nx is line j-1, the
 * reference's naming in poisson.f90:42):
 *   y(i,j) = c x(idx) - ( wl x(idx-1) + wr x(idx+1) + wd x(idx+nx) + wu x(idx-nx) ),   missing neighbours = 0
 * evaluation order (every kernel, and the same as KL_OP_ANISO5_VAR's):
 *   s = fma(wl, xl, wr*xr) ; t = fma(wd, xd, wu*xu) ; y = fma(c, xc, -(s + t))
 * so c = ((a+a)+b)+b, wl = wr = a, wd = wu = b gives KL_OP_ANISO5_VAR on constant fields kx = a, ky = b bit for bit.
 * Convection-diffusion -lap(u) + (bx, by).grad(u) on a grid of spacing h, scaled by h^2, with the cell Peclet numbers
 * px = bx*h/2, py = by*h/2: central differences c = 4, wl = 1+px, wr = 1-px, wu = 1+py, wd = 1-py (real spectrum iff
 * |px|, |py| <= 1); first-order upwind (px, py >= 0) c = 4+2px+2py, wl = 1+2px, wr = 1, wu = 1+2py, wd = 1.           */
typedef struct {
    double c, wl, wr, wd, wu;
} kl_stencil5_t;
/* Exact extremes of the Dirichlet spectrum of KL_OP_STENCIL5 on an nx x ny grid (host arithmetic, no handle).  When
 * wl*wr >= 0 and wd*wu >= 0 the operator is similar to a symmetric one by a diagonal scaling and its spectrum is real:
 *   lambda = c -+ 2 sqrt(wl*wr) cos(pi/(nx+1)) -+ 2 sqrt(wd*wu) cos(pi/(ny+1))
 * (KL_OK).  Otherwise the spectrum is complex: KL_ERR_UNSUPPORTED and both outputs NaN.  Pass [lam_min, lam_max] to
 * KL_PC_CHEB as its interval.                                                                                         */
int kl_stencil5_spectrum(const kl_stencil5_t *w, int nx, int ny, double *lam_min, double *lam_max);
typedef struct {
    int kind;
    double eps_x, eps_y;  /* KL_OP_ANISO5 */
    kl_apply_fn fn;       /* KL_OP_USER   */
    void *user;
} kl_operator_t;

/* ---- preconditioner plug-in: replaces procedure(precond) ----------------
 * src/interfaces.f90:19-28   subroutine precond(A_x, r, z, aux, params, n)  */
typedef int (*kl_precond_fn)(kl_handle_t h, const kl_operator_t *A_x, void *user,
                             const double *d_r, double *d_z, double *d_aux, const double *params,
                             int nparams, int nx, int ny_local, void *cuda_stream);
enum {
    KL_PC_NONE = 0,
    KL_PC_CBPR2 = 1,  /* chebyshev_precond::cbpr2  src/preconds/chebyshev.f90:8-38 */
    KL_PC_CHEB = 2,   /* degree-k Chebyshev iteration (new; README.md:11)          */
    KL_PC_JACOBI_CHEB = 3, /* degree-k Chebyshev iteration on the Jacobi-scaled operator D^-1 A, D = diag(A), for
                          KL_OP_ANISO5_VAR only (new).  degree 0: z = D^-1 r (point Jacobi), params ignored; degree
                          k >= 1: params = (a, b), an interval of the spectrum of D^-1 A in either order.  That
                          spectrum lies in (0, 2] for every positive coefficient field (Gershgorin: the off-diagonal
                          row sums of A are at most its diagonal), so b = 2 needs no estimate, and
                          kl_cheb_interval_from_ritz(2.0 / 1.025, k) yields (2, 2/ratio(k)) from the measured ratio
                          table.  Degree k <= 6 runs as ONE temporally blocked pass (r, kx, ky in, z out: 32n B)
                          on even nx >= 64 with KL_OPT_TMA, KL_OPT_FUSE and KL_OPT_CHAIN on; otherwise, and for
                          the steps beyond the sixth, one pass per step.  Constant-diagonal operators use
                          KL_PC_CHEB with the interval scaled by their diagonal.                              */
    KL_PC_USER = 100
};
typedef struct {
    int kind;
    int degree;        /* KL_PC_CHEB, KL_PC_JACOBI_CHEB */
    kl_precond_fn fn;  /* KL_PC_USER */
    void *user;
} kl_precond_t;

/* ---- lifecycle --------------------------------------------------------- */
int kl_create(kl_handle_t *h, int device);
int kl_destroy(kl_handle_t h);
const char *kl_last_error(kl_handle_t h);
int kl_version(void);
/* use an existing CUDA stream (e.g. torch's current stream; pass cudaStreamLegacy = (void*)1 for the legacy default
 * stream); NULL = the handle's own non-blocking stream.  In device-pointer mode the caller's vectors must be
 * ordered against the handle's stream: either share the stream that produces / consumes them, or synchronise. */
int kl_set_stream(kl_handle_t h, void *cuda_stream);
/* the stream the handle enqueues on (for event-based ordering against the caller's own streams) */
int kl_get_stream(kl_handle_t h, void **cuda_stream);
int kl_synchronize(kl_handle_t h);

enum { KL_POINTER_HOST = 0, KL_POINTER_DEVICE = 1 };
int kl_set_pointer_mode(kl_handle_t h, int mode);

/* options */
enum {
    KL_OPT_ORTHO = 1,         /* GMRES-MGSR orthogonalisation, see below             */
    KL_OPT_MAX_RESTARTS = 2,  /* default 1000 = max_restarts (gmres_mgsr.f90:6) / stages (gmres_hh.f90:8) */
    KL_OPT_VERR = 3,          /* 1 (default): compute the v_err epilogue; 0: skip it */
    KL_OPT_CHECK_EVERY = 4,   /* CG/BiCGSTAB: iterations enqueued between host polls (default 32) */
    KL_OPT_USE_GRAPH = 5,     /* reserved (CUDA-graph replay of an iteration batch); currently a no-op */
    KL_OPT_HH_MODE = 6,       /* Householder application, see below                  */
    KL_OPT_FUSE = 7,          /* 1 (default): fused kernels; 0: one kernel per reference loop */
    KL_OPT_PROFILE = 8,       /* 1: CUDA-event pairs around every hot kernel (kl_get_profile)  */
    KL_OPT_TMA = 9,           /* 1 (default): TMA-staged stencil kernels; 0: register-pipelined ones */
    KL_OPT_REORTH_ETA = 11,   /* KL_ORTHO_CGS2_SELECTIVE threshold eta in 1/1000 (default 300; 707 = 1/sqrt2 is the classical bound):
                                 the second Gram-Schmidt pass runs only when ||w'|| < eta ||w||          */
    KL_OPT_CHAIN = 12,        /* 1 (default): temporally blocked kernels -- several dependent operator applications
                                 (Chebyshev degree k, cbpr2 o A, A o cbpr2) in one pass over HBM; 0: one pass each */
    KL_OPT_STENCIL_ROWS = 13, /* grid lines per CTA of the temporally blocked kernels (0 = heuristic)       */
    KL_OPT_INLINE_ALLREDUCE = 14, /* multi-GPU with peer memory: 1 (default) = the last block of a reducing kernel does
                                 the NVLink all-reduce and the scalar recurrence itself; 0 = separate kernels  */
    KL_OPT_PDL = 15,          /* 1 (default): the fused CG kernels and, on one GPU, every kernel of a GMRES / Householder
                                 restart cycle are launched with programmatic dependent launch, so the launch and
                                 prologue of one overlap the tail of the other; 0: plain stream order            */
    KL_OPT_STENCIL_TAIL = 17, /* lines per CTA in the tapered tail of the stencil kernels' grids: -1 (default) = a quarter
                                 of the regular tile height, 0 = off                                            */
    KL_OPT_STENCIL_STAGGER = 18, /* 1: CTA heights of the stencil kernels staggered (5/8 .. 11/8 of the mean) so that CTAs
                                 do not start and drain in lockstep waves; 0 (default): equal heights -- measured
                                 neutral on B200 (profiles/r02_cta_timeline.md)                                   */
    KL_OPT_REVERSE = 19,      /* 1: the second kernel of a CG iteration marches the grid from its last lines to its first,
                                 i.e. starts on what the first kernel left in L2; 0 (default): measured neutral     */
    KL_OPT_COOP = 20,         /* 1: on small grids (launch-bound, basis resident in L2) the three passes of the CGS2
                                 orthogonalisation run as ONE cooperative kernel with two grid barriers; 0 (default):
                                 three graph-replayed launches measured 4 % faster at 300^2                         */
    KL_OPT_PERSISTENT = 21,   /* 1: the TMA stencil kernels run persistent CTAs (as many as fit on the GPU) that loop over
                                 the tiles with the TMA ring running across tile boundaries; 0 (default) = one CTA per
                                 tile -- the hardware's dynamic CTA scheduling balances better (measured)            */
    KL_OPT_CG_ONEPASS = 22,   /* plain CG on one GPU with a built-in 5-point operator: 1 = one temporally blocked pass per
                                 iteration (48n B, one reduction; beta predicted from three dot products of the same
                                 pass), 2 = pairs of such passes that store p and x every second iteration only (36n B,
                                 bit-identical to 1), 0 = two stencil passes (64n B), -1 (default) = one pass from 2^20
                                 unknowns on (1.3-1.8x faster there on B200; smaller grids, which fit in L2, keep two
                                 passes), pairs from 2^24 on                                                          */
    KL_OPT_X0 = 23,           /* solver entries (not kl_lanczos): 0 (default) = x is output only and the solve starts from
                                 x = 0, as the reference does; 1 = x is read on entry as the initial guess x0 and
                                 overwritten with the solution (host mode: the nx*ny doubles at x are uploaded and
                                 counted in h2d_bytes; device mode: x is used in place and must not be b).  CG, PCG and
                                 BiCGSTAB start from r0 = b - A x0 with the same absolute test ||r|| < tol; GMRES and
                                 Householder GMRES start their first cycle from x0 and keep final_err = |g_j+1|/||b||;
                                 iter, n_out, restart_out / stages_out and the history count this call only.  If the
                                 initial residual norm of the stopping test (||r0||, or ||M^-1 (b - A x0)|| / ||b||
                                 for GMRES) is below tol or zero, the call returns KL_OK at once with x = x0 untouched,
                                 iter = 0 and res = ||r0|| (GMRES: n_out = 0, restart_out = 1, final_err = v_err = 0)
                                 and an empty history.  One GPU only (KL_ERR_UNSUPPORTED on a multi-GPU handle); no
                                 environment variable.                                                           */
    KL_OPT_PUSH_HALO = 16,    /* multi-GPU with peer memory: 1 (default) = the kernel that PRODUCES a vector pushes its
                                 boundary lines into the neighbours' halo slots (no halo kernel; the all-reduce that
                                 ends the kernel is the barrier); 0 = separate halo push before every operator apply */
    KL_OPT_PEER = 10          /* multi-GPU: 1 = NVLink peer-memory all-reduce / halo push (default when the
                                 IPC mapping succeeded), 0 = NCCL collectives.  Set on all ranks alike. */
};
enum {
    KL_ORTHO_MGS2 = 0,  /* the reference's modified Gram-Schmidt applied twice (gmres_mgsr.f90:341-360) */
    KL_ORTHO_CGS2 = 1,  /* classical Gram-Schmidt twice: h = V^T w one-pass kernels (default)           */
    KL_ORTHO_CGS2_SELECTIVE = 2 /* CGS with the second update only when ||w'|| < eta ||w|| (device-side test) */
};
enum {
    KL_HH_SEQUENTIAL = 0, /* reflector by reflector, the reference's order (gmres_hh.f90:269-304) */
    KL_HH_BLOCKED = 1     /* compact-WY, three tall-skinny passes per step (default when n >= 4096, m <= 96) */
};
int kl_set_option(kl_handle_t h, int key, int value);
int kl_get_option(kl_handle_t h, int key, int *value);

/* ---- multi-GPU: one process per GPU, row-slab decomposition -------------- */
#define KL_UNIQUE_ID_BYTES 128
int kl_comm_unique_id(void *id_out /* KL_UNIQUE_ID_BYTES */);
int kl_comm_init(kl_handle_t h, int rank, int nranks, const void *id /* same bytes on all ranks */);
int kl_comm_rank(kl_handle_t h, int *rank, int *nranks);
/* lines [j0, j0+ny_local) of a global nx*ny grid owned by this handle's rank */
int kl_partition(kl_handle_t h, int ny, int *j0, int *ny_local);
/* the same rule without a handle: contiguous lines, the first ny % nranks ranks get one more */
int kl_partition_rank(int ny, int rank, int nranks, int *j0, int *ny_local);

/* ---- device vectors (so that b/x can stay resident between calls) -------- */
int kl_vec_alloc(kl_handle_t h, size_t n, double **d_ptr);
int kl_vec_free(kl_handle_t h, double *d_ptr);
int kl_vec_upload(kl_handle_t h, double *d_dst, const double *h_src, size_t n);
int kl_vec_download(kl_handle_t h, double *h_dst, const double *d_src, size_t n);

/* ---- operator / preconditioner application ------------------------------
 * call stvec(x, y, n)                      src/problems/poisson.f90:33
 * call cbpr2(A_x, r, z, aux, params, n)    src/preconds/chebyshev.f90:8
 * Host pointer mode: the vectors are copied in and out and the call returns when y / z is on the host.
 * Device pointer mode: x / r and y / z (distinct buffers) are used in place and the call is stream-ordered
 * (it returns after enqueueing; kl_synchronize or any later call on the handle's stream orders after it).
 * KL_PC_CHEB of degree k <= 12 runs as one or two temporally blocked passes over HBM (KL_OPT_CHAIN).      */
int kl_apply_operator(kl_handle_t h, const kl_operator_t *A_x, const double *x, double *y, int nx,
                      int ny);
int kl_apply_precond(kl_handle_t h, const kl_precond_t *M_inv, const kl_operator_t *A_x,
                     const double *r, double *z, const double *params, int nparams, int nx,
                     int ny);

/* ---- solvers -------------------------------------------------------------
 * Output sizes: x[nx*ny_local], final_err[m], v_err[m+1].
 * x is output only unless KL_OPT_X0 = 1, which makes it the initial guess as well.   */

/* gmres_mgsr_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,restart_out,M_inv,params)
 * src/gmres_mgsr.f90:277 */
int kl_gmres_mgsr_omp(kl_handle_t h, const kl_operator_t *Ax_vec, const double *b, double *x,
                      int nx, int ny, int m, double tol, double *final_err, double *v_err,
                      int *n_out, int *restart_out, const kl_precond_t *M_inv,
                      const double *params, int nparams);
/* gmres_mgsr_mf(...) same list, serial twin with in-cycle early exit
 * src/gmres_mgsr.f90:98 */
int kl_gmres_mgsr_mf(kl_handle_t h, const kl_operator_t *Ax_vec, const double *b, double *x,
                     int nx, int ny, int m, double tol, double *final_err, double *v_err,
                     int *n_out, int *restart_out, const kl_precond_t *M_inv,
                     const double *params, int nparams);
/* gmres_hh_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,stages_out)
 * src/gmres_hh.f90:211 */
int kl_gmres_hh_omp(kl_handle_t h, const kl_operator_t *Ax_vec, const double *b, double *x, int nx,
                    int ny, int m, double tol, double *final_err, double *v_err, int *n_out,
                    int *stages_out);
/* gmres_hh_prec_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,stages_out,m_inv,params)
 * src/gmres_hh.f90:388 */
int kl_gmres_hh_prec_omp(kl_handle_t h, const kl_operator_t *Ax_vec, const double *b, double *x,
                         int nx, int ny, int m, double tol, double *final_err, double *v_err,
                         int *n_out, int *stages_out, const kl_precond_t *m_inv,
                         const double *params, int nparams);
/* ---- dense-operator variants (small n: O(n^2) storage) ------------------------------------
 * A is the Fortran array A(n,n): column-major, leading dimension n; host or device pointer
 * according to kl_set_pointer_mode (a host matrix is copied to the device inside the call).
 * w = matmul(A, v) is evaluated as the column sweep y(:) = y(:) + A(:,j)*v(j), j = 1..n (every
 * y(i) a sequential FMA sum over j).  Semantics: in-cycle exit on h_val < tol or
 * final_err(j) < tol, no preconditioner.
 * gmres_mgsr_dense(A,b,x,m,tol,final_err,v_err,n_out,restart_out)   src/gmres_mgsr.f90:11-95  */
int kl_gmres_mgsr_dense(kl_handle_t h, const double *A, int n, const double *b, double *x, int m, double tol,
                        double *final_err, double *v_err, int *n_out, int *restart_out);
/* gmres_hh_dense(A,b,x,m,tol,final_err,v_err,n_out,stages_out)       src/gmres_hh.f90:10-112
 * (m <= n: m = n takes the reference's `if (j < n)` else-branch at the last step; m > n indexes v_j(j) out of
 * bounds in the reference itself and is rejected)                                                  */
int kl_gmres_hh_dense(kl_handle_t h, const double *A, int n, const double *b, double *x, int m, double tol,
                      double *final_err, double *v_err, int *n_out, int *stages_out);
/* hilbert::generate_matrix(H, n)  src/problems/hilbert.f90:6-18: H(i,j) = 1/real(i+j-1), the quotient
 * in SINGLE precision (default real) widened to double, as the reference computes it.          */
int kl_generate_matrix(kl_handle_t h, double *H, int n);
/* y = matmul(A, x) (the drivers build b = matmul(A, 1) this way, tests/test_hilbert.f90:44-45) */
int kl_dense_matvec(kl_handle_t h, const double *A, int n, const double *x, double *y);

/* cg(Ax_op,b,x,tol,iter,res) src/cg.f90:11 ; cg_omp(...) src/cg.f90:83
 * iter: maximum on entry, count on exit (unchanged if not converged).        */
int kl_cg(kl_handle_t h, const kl_operator_t *Ax_op, const double *b, double *x, int nx, int ny,
          double tol, int *iter, double *res);
int kl_cg_omp(kl_handle_t h, const kl_operator_t *Ax_op, const double *b, double *x, int nx,
              int ny, double tol, int *iter, double *res);
/* pcg(Ax_op,b,x,tol,iter,res,M_inv,params) src/cg.f90:44 ; pcg_omp src/cg.f90:154 */
int kl_pcg(kl_handle_t h, const kl_operator_t *Ax_op, const double *b, double *x, int nx, int ny,
           double tol, int *iter, double *res, const kl_precond_t *M_inv, const double *params,
           int nparams);
int kl_pcg_omp(kl_handle_t h, const kl_operator_t *Ax_op, const double *b, double *x, int nx,
               int ny, double tol, int *iter, double *res, const kl_precond_t *M_inv,
               const double *params, int nparams);
/* bicgstab(ax_op,b,x,tol,iter,res) src/bicgstab.f90:12 */
int kl_bicgstab(kl_handle_t h, const kl_operator_t *ax_op, const double *b, double *x, int nx,
                int ny, double tol, int *iter, double *res);
/* pbicgstab(ax_op,b,x,tol,iter,res,m_inv,params) src/bicgstab.f90:49 */
int kl_pbicgstab(kl_handle_t h, const kl_operator_t *ax_op, const double *b, double *x, int nx,
                 int ny, double tol, int *iter, double *res, const kl_precond_t *m_inv,
                 const double *params, int nparams);
/* pbicgstab_omp(ax_op,b,x,tol,max_iter,res,m_inv,params) src/bicgstab.f90:91 */
int kl_pbicgstab_omp(kl_handle_t h, const kl_operator_t *ax_op, const double *b, double *x, int nx,
                     int ny, double tol, int *max_iter, double *res, const kl_precond_t *m_inv,
                     const double *params, int nparams);

/* ---- Lanczos spectral estimate (README.md:11; no reference code) ---------
 * k-step Lanczos on A started from b/||b||, b = A*1; returns the extreme Ritz
 * values.  kl_cheb_params_from_ritz applies the reference drivers' literal
 * policy (8.2, 0.2) = (1.025*lambda_max, 1.025*lambda_max/41) to an estimate. */
int kl_lanczos(kl_handle_t h, const kl_operator_t *A_x, int nx, int ny, int steps,
               double *theta_min, double *theta_max);
int kl_cheb_params_from_ritz(double theta_min, double theta_max, double params_out[2]);
/* interval [b/ratio(degree), b], b = 1.025*theta_max, for KL_PC_CHEB of the given degree (ratios from the
 * measured sweep profiles/r01_cheb_sweep_2048.json: 41, 100, 400, 400, 1000, ...)                        */
int kl_cheb_interval_from_ritz(double theta_max, int degree, double params_out[2]);

/* ---- diagnostics of the last solver call --------------------------------- */
/* residual estimate of every inner iteration across restarts (final_err for
 * GMRES, ||r||_2 for CG/BiCGSTAB).  *len = number recorded (may exceed cap).   */
int kl_get_history(kl_handle_t h, double *out, int cap, int *len);
typedef struct {
    int iterations;          /* total inner iterations of the last solve          */
    int cycles;              /* GMRES restart cycles / host polls                  */
    double solve_ms;         /* CUDA-event time of the iteration loop (no H2D/D2H) */
    double total_ms;         /* including host<->device copies                     */
    double algorithmic_bytes;/* minimum-traffic bytes of the executed kernels      */
    long long kernel_launches;
    double orth_frobenius;   /* ||I - V^T V||_F of the last basis when KL_OPT_VERR */
    double h2d_bytes, d2h_bytes;
    int reorth_skipped;      /* KL_ORTHO_CGS2_SELECTIVE: second passes skipped            */
} kl_stats_t;
int kl_get_stats(kl_handle_t h, kl_stats_t *out);
/* per-kernel-class timers of the last solve (KL_OPT_PROFILE = 1): class idx in
 * [0, KL_PROFILE_CLASSES); name may be NULL.  Returns KL_ERR_INVALID past the end. */
#define KL_PROFILE_CLASSES 8
int kl_get_profile(kl_handle_t h, int idx, const char **name, double *ms, long long *launches,
                   double *algorithmic_bytes);

#ifdef __cplusplus
}
#endif
#endif /* KRYLOV_B200_H */
