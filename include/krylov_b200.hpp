// krylov_b200.hpp -- C++ host-side mirror of the reference's module procedures on top of
// the C ABI (krylov_b200.h).  Header-only; link with -lkrylov_b200.
//
// The reference is Fortran and no Fortran compiler exists in the build image, so the
// drivers that exercise the library natively (drivers/*.cpp) are written in C++ against
// this header.  Names, argument order and intent follow the Fortran interfaces:
//
//   gmres_mgsr_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,restart_out,M_inv,params)  src/gmres_mgsr.f90:277
//   gmres_mgsr_mf (same list)                                                        src/gmres_mgsr.f90:98
//   gmres_hh_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,stages_out)                  src/gmres_hh.f90:211
//   gmres_hh_prec_omp(...,m_inv,params)                                              src/gmres_hh.f90:388
//   cg / cg_omp(Ax_op,b,x,tol,iter,res)                                              src/cg.f90:11 / :83
//   pcg / pcg_omp(...,M_inv,params)                                                  src/cg.f90:44 / :154
//   bicgstab / pbicgstab / pbicgstab_omp                                             src/bicgstab.f90:12 / :49 / :91
//   stvec(x,y,n) / stv_poisson(x,y,n)                                                src/problems/poisson.f90:33 / :79
//   cbpr2(A_x,r,z,aux,params,n)                                                      src/preconds/chebyshev.f90:8
//
// `allocatable, intent(out)` arrays (x, final_err, v_err) are std::vector<double>& that the
// callee resizes -- the reference's "callee allocates" ownership.  The operator and the
// preconditioner are passed as descriptors (kl_operator_t / kl_precond_t) instead of
// procedure arguments; krylov::stvec, krylov::stv_poisson and krylov::cbpr2 name the built-ins.
#pragma once
#include <cmath>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "krylov_b200.h"

namespace krylov {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

inline const kl_operator_t stvec{KL_OP_POISSON5, 1.0, 1.0, nullptr, nullptr};
inline const kl_operator_t stv_poisson{KL_OP_POISSON5_BRANCHY, 1.0, 1.0, nullptr, nullptr};
inline kl_operator_t aniso(double ex, double ey) { return kl_operator_t{KL_OP_ANISO5, ex, ey, nullptr, nullptr}; }
// general constant-coefficient 5-point operator (KL_OP_STENCIL5, krylov_b200.h kl_stencil5_t).  It converts to the
// kl_operator_t every entry takes; that descriptor points at this object's weights, so the object must outlive the
// calls it is passed to.
struct stencil5 {
    kl_stencil5_t w;
    kl_operator_t op;
    stencil5(double c, double wl, double wr, double wd, double wu)
        : w{c, wl, wr, wd, wu}, op{KL_OP_STENCIL5, 1.0, 1.0, nullptr, &w} {}
    stencil5(const stencil5 &o) : stencil5(o.w.c, o.w.wl, o.w.wr, o.w.wd, o.w.wu) {}
    stencil5 &operator=(const stencil5 &o) { w = o.w; return *this; }
    operator const kl_operator_t &() const { return op; }
    // exact extremes of the spectrum on an nx x ny grid (kl_stencil5_spectrum); throws if it is complex
    std::pair<double, double> spectrum(int nx, int ny) const {
        double lo, hi;
        const int rc = kl_stencil5_spectrum(&w, nx, ny, &lo, &hi);
        if (rc != KL_OK) throw Error(rc, "kl_stencil5_spectrum: complex spectrum (wl*wr < 0 or wd*wu < 0) or bad arguments");
        return {lo, hi};
    }
};
// sparse n x n matrix in CSR form (KL_OP_CSR, krylov_b200.h kl_csr_t): row_ptr, col_ind and val are DEVICE arrays of
// n+1, nnz and nnz entries.  Pass nx = n, ny = 1.  Like stencil5, the descriptor points at this object, which must
// outlive the calls it is passed to.
struct csr {
    kl_csr_t m;
    kl_operator_t op;
    csr(int64_t nnz, const int64_t *row_ptr, const int32_t *col_ind, const double *val)
        : m{nnz, row_ptr, col_ind, val}, op{KL_OP_CSR, 1.0, 1.0, nullptr, &m} {}
    csr(const csr &o) : csr(o.m.nnz, o.m.row_ptr, o.m.col_ind, o.m.val) {}
    csr &operator=(const csr &o) { m = o.m; return *this; }
    operator const kl_operator_t &() const { return op; }
};
inline const kl_precond_t cbpr2{KL_PC_CBPR2, 0, nullptr, nullptr};
inline const kl_precond_t no_precond{KL_PC_NONE, 0, nullptr, nullptr};
inline kl_precond_t cheb(int degree) { return kl_precond_t{KL_PC_CHEB, degree, nullptr, nullptr}; }
// Chebyshev on the Jacobi-scaled operator D^-1 A (variable-coefficient and CSR operators only; degree 0 = point Jacobi)
inline kl_precond_t jacobi_cheb(int degree) { return kl_precond_t{KL_PC_JACOBI_CHEB, degree, nullptr, nullptr}; }

class Handle {
public:
    explicit Handle(int device = 0) {
        int rc = kl_create(&h_, device);
        if (rc != KL_OK) throw Error(rc, "kl_create failed: no usable CUDA device (there is no CPU fallback)");
    }
    ~Handle() { kl_destroy(h_); }
    Handle(const Handle &) = delete;
    Handle &operator=(const Handle &) = delete;
    kl_handle_t get() const { return h_; }
    void set_option(int key, int value) { check(kl_set_option(h_, key, value)); }
    int check(int rc) const {
        if (rc < 0) throw Error(rc, std::string("libkrylov_b200: ") + kl_last_error(h_));
        return rc;
    }
    kl_stats_t stats() const {
        kl_stats_t s;
        kl_get_stats(h_, &s);
        return s;
    }
    std::vector<double> history() const {
        int n = 0;
        kl_get_history(h_, nullptr, 0, &n);
        std::vector<double> v(n > 0 ? n : 0);
        if (n > 0) kl_get_history(h_, v.data(), n, &n);
        return v;
    }

private:
    kl_handle_t h_ = nullptr;
};

// nsize = int(sqrt(real(n)))  -- single precision, as in the reference (gmres_mgsr.f90:298)
inline int grid_side(size_t n) { return (int)std::sqrt((float)n); }

// call stvec(x, y, n)
inline void apply(Handle &h, const kl_operator_t &A, const std::vector<double> &x, std::vector<double> &y, int n) {
    y.resize(x.size());
    h.check(kl_apply_operator(h.get(), &A, x.data(), y.data(), n, (int)(x.size() / n)));
}
// call cbpr2(A_x, r, z, aux, params, n)   (aux is library-owned scratch)
inline void apply_precond(Handle &h, const kl_precond_t &M, const kl_operator_t &A, const std::vector<double> &r,
                          std::vector<double> &z, const std::vector<double> &params, int n) {
    z.resize(r.size());
    h.check(kl_apply_precond(h.get(), &M, &A, r.data(), z.data(), params.data(), (int)params.size(), n,
                             (int)(r.size() / n)));
}

inline int gmres_mgsr_omp(Handle &h, const kl_operator_t &Ax_vec, const std::vector<double> &b, std::vector<double> &x,
                          int m, double tol, std::vector<double> &final_err, std::vector<double> &v_err, int &n_out,
                          int &restart_out, const kl_precond_t &M_inv, const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_mgsr_omp(h.get(), &Ax_vec, b.data(), x.data(), ns, ns, m, tol, final_err.data(), v_err.data(),
                                     &n_out, &restart_out, &M_inv, params.data(), (int)params.size()));
}
inline int gmres_mgsr_mf(Handle &h, const kl_operator_t &Ax_vec, const std::vector<double> &b, std::vector<double> &x,
                         int m, double tol, std::vector<double> &final_err, std::vector<double> &v_err, int &n_out,
                         int &restart_out, const kl_precond_t &M_inv, const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_mgsr_mf(h.get(), &Ax_vec, b.data(), x.data(), ns, ns, m, tol, final_err.data(), v_err.data(),
                                    &n_out, &restart_out, &M_inv, params.data(), (int)params.size()));
}
inline int gmres_hh_omp(Handle &h, const kl_operator_t &Ax_vec, const std::vector<double> &b, std::vector<double> &x,
                        int m, double tol, std::vector<double> &final_err, std::vector<double> &v_err, int &n_out,
                        int &stages_out) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_hh_omp(h.get(), &Ax_vec, b.data(), x.data(), ns, ns, m, tol, final_err.data(), v_err.data(),
                                   &n_out, &stages_out));
}
inline int gmres_hh_prec_omp(Handle &h, const kl_operator_t &Ax_vec, const std::vector<double> &b,
                             std::vector<double> &x, int m, double tol, std::vector<double> &final_err,
                             std::vector<double> &v_err, int &n_out, int &stages_out, const kl_precond_t &m_inv,
                             const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_hh_prec_omp(h.get(), &Ax_vec, b.data(), x.data(), ns, ns, m, tol, final_err.data(),
                                        v_err.data(), &n_out, &stages_out, &m_inv, params.data(), (int)params.size()));
}
// ---- dense-operator variants: A is column-major n x n (A[i + j*n] = A(i,j)) like the Fortran array ----
// gmres_mgsr_dense(A,b,x,m,tol,final_err,v_err,n_out,restart_out)   src/gmres_mgsr.f90:11
inline int gmres_mgsr_dense(Handle &h, const std::vector<double> &A, const std::vector<double> &b, std::vector<double> &x,
                            int m, double tol, std::vector<double> &final_err, std::vector<double> &v_err, int &n_out,
                            int &restart_out) {
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_mgsr_dense(h.get(), A.data(), (int)b.size(), b.data(), x.data(), m, tol, final_err.data(),
                                       v_err.data(), &n_out, &restart_out));
}
// gmres_hh_dense(A,b,x,m,tol,final_err,v_err,n_out,stages_out)       src/gmres_hh.f90:10
inline int gmres_hh_dense(Handle &h, const std::vector<double> &A, const std::vector<double> &b, std::vector<double> &x,
                          int m, double tol, std::vector<double> &final_err, std::vector<double> &v_err, int &n_out,
                          int &stages_out) {
    x.assign(b.size(), 0.0); final_err.assign(m, 0.0); v_err.assign(m + 1, 0.0);
    return h.check(kl_gmres_hh_dense(h.get(), A.data(), (int)b.size(), b.data(), x.data(), m, tol, final_err.data(),
                                     v_err.data(), &n_out, &stages_out));
}
// generate_matrix(H, n)   src/problems/hilbert.f90:6   (callee allocates)
inline void generate_matrix(Handle &h, std::vector<double> &H, int n) {
    H.assign((size_t)n * n, 0.0);
    h.check(kl_generate_matrix(h.get(), H.data(), n));
}
// b = matmul(A, x)
inline void matmul(Handle &h, const std::vector<double> &A, const std::vector<double> &x, std::vector<double> &y) {
    y.assign(x.size(), 0.0);
    h.check(kl_dense_matvec(h.get(), A.data(), (int)x.size(), x.data(), y.data()));
}
// iter: maximum on entry, count on exit (unchanged if not converged) -- cg.f90:15
inline int cg_omp(Handle &h, const kl_operator_t &Ax_op, const std::vector<double> &b, std::vector<double> &x, double tol,
                  int &iter, double &res) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_cg_omp(h.get(), &Ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res));
}
inline int cg(Handle &h, const kl_operator_t &Ax_op, const std::vector<double> &b, std::vector<double> &x, double tol,
              int &iter, double &res) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_cg(h.get(), &Ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res));
}
inline int pcg_omp(Handle &h, const kl_operator_t &Ax_op, const std::vector<double> &b, std::vector<double> &x, double tol,
                   int &iter, double &res, const kl_precond_t &M_inv, const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_pcg_omp(h.get(), &Ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res, &M_inv, params.data(),
                              (int)params.size()));
}
inline int pcg(Handle &h, const kl_operator_t &Ax_op, const std::vector<double> &b, std::vector<double> &x, double tol,
               int &iter, double &res, const kl_precond_t &M_inv, const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_pcg(h.get(), &Ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res, &M_inv, params.data(),
                          (int)params.size()));
}
inline int bicgstab(Handle &h, const kl_operator_t &ax_op, const std::vector<double> &b, std::vector<double> &x,
                    double tol, int &iter, double &res) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_bicgstab(h.get(), &ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res));
}
inline int pbicgstab(Handle &h, const kl_operator_t &ax_op, const std::vector<double> &b, std::vector<double> &x,
                     double tol, int &iter, double &res, const kl_precond_t &m_inv, const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_pbicgstab(h.get(), &ax_op, b.data(), x.data(), ns, ns, tol, &iter, &res, &m_inv, params.data(),
                                (int)params.size()));
}
inline int pbicgstab_omp(Handle &h, const kl_operator_t &ax_op, const std::vector<double> &b, std::vector<double> &x,
                         double tol, int &max_iter, double &res, const kl_precond_t &m_inv,
                         const std::vector<double> &params) {
    const int ns = grid_side(b.size());
    x.assign(b.size(), 0.0);
    return h.check(kl_pbicgstab_omp(h.get(), &ax_op, b.data(), x.data(), ns, ns, tol, &max_iter, &res, &m_inv,
                                    params.data(), (int)params.size()));
}

}  // namespace krylov
