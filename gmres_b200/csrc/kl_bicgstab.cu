// kl_bicgstab.cu -- BiCGSTAB, plain and right-preconditioned.
//
// Reference: src/bicgstab.f90  bicgstab :12-47, pbicgstab :49-89, pbicgstab_omp :91-182.
// (The serial variants leave the loop before the beta/p update, the OpenMP one
// finishes the iteration and skips the rest: same x, same count.)
//
// Fused path, built-in operator, per iteration:
//  no preconditioner (136n B):
//   K1  p' = r + beta (p - omega ap) ; ap' = A p' ; ap'.r0      reads r,p,ap,r0  writes p',ap'  48n
//   K2  s = r - alpha ap' ; as = A s ; as.s, as.as              reads r,ap'      writes s,as    32n
//   K3  x += alpha p' + omega s ; r = s - omega as ; r.r, r.r0  reads x,p',s,as,r0 writes x,r   56n
//  cbpr2 (160n B): K1/K2 are temporally blocked chains (kl_chain_tma.cuh): direction update, cbpr2 and the
//   operator in one pass (ChBiDir 56n, ChBiS 40n), K3 64n.  KL_OPT_CHAIN = 0 (184n B): K1/K2
//   produce z1 = cbpr2(p'), z2 = cbpr2(s) in one pass and a second stencil kernel applies the operator to
//   z1/z2 carrying the dot products.
// p and ap are ping-ponged because neighbouring thread blocks still read the old
// values while the new ones are written.
#include <math.h>

#include "kl_ops.cuh"

namespace kl {

// K1: direction update fused into the operator (CB = false) or into cbpr2 (CB = true)
template <bool CB>
struct FBiDir : StencilBase<3, (CB ? 0 : 1)> {
    double *p_new, *out;   // out = ap' (CB = false) or z1 (CB = true)
    const double *r0;
    const double *S;
    double beta, omega, d, calpha;
    FastDiv fd;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];
        omega = S[S_OMEGA];
        fd.set(d);
    }
    __device__ __forceinline__ double pn(double r, double p, double ap) const {
        return fma(beta, fma(-omega, ap, p), r);     // bicgstab.f90:176
    }
    __device__ __forceinline__ double point(const double (&v)[3]) const {
        const double t = pn(v[0], v[1], v[2]);
        return CB ? fd.div(t) : t;
    }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[3][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
        if (CB) {
            double pv[VEC], zv[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                pv[v] = pn(raw[0][v], raw[1][v], raw[2][v]);
                zv[v] = fma(calpha, pv[v] - au[v], cu[v]);   // chebyshev.f90:35
            }
            KL_ST(VEC, p_new, idx, pv)
            KL_ST(VEC, out, idx, zv)
        } else {
            double q[VEC];
            KL_LD(VEC, q, r0, idx)
            KL_ST(VEC, p_new, idx, cu)
            KL_ST(VEC, out, idx, au)
#pragma unroll
            for (int v = 0; v < VEC; ++v) acc[0] = fma(au[v], q[v], acc[0]);   // :126
        }
    }
};

// K2: s = r - alpha ap fused into the operator (CB = false) or into cbpr2 (CB = true)
template <bool CB>
struct FBiS : StencilBase<2, (CB ? 0 : 2)> {
    double *s, *out;       // out = as (CB = false) or z2 (CB = true)
    const double *S;
    double alpha, d, calpha;
    FastDiv fd;
    __device__ __forceinline__ void init() { alpha = S[S_ALPHA]; fd.set(d); }
    __device__ __forceinline__ double point(const double (&v)[2]) const {
        const double t = fma(-alpha, v[1], v[0]);    // bicgstab.f90:134
        return CB ? fd.div(t) : t;
    }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[2][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
        if (CB) {
            double sv[VEC], zv[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                sv[v] = fma(-alpha, raw[1][v], raw[0][v]);
                zv[v] = fma(calpha, sv[v] - au[v], cu[v]);
            }
            KL_ST(VEC, s, idx, sv)
            KL_ST(VEC, out, idx, zv)
        } else {
            KL_ST(VEC, s, idx, cu)
            KL_ST(VEC, out, idx, au)
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                acc[0] = fma(au[v], cu[v], acc[0]);  // :141 as.s
                acc[1] = fma(au[v], au[v], acc[1]);  // :142 as.as
            }
        }
    }
};

// ---- temporally blocked variants for cbpr2 (kl_chain_tma.cuh): preconditioner and operator in ONE pass ----
// K1: p' = r + beta (p - omega ap) ; z1 = cbpr2(p') ; ap' = A z1 ; ap'.r0
//     reads r,p,ap,r0  writes p',z1,ap'  (56n B instead of 40n + 24n)
struct ChBiDir : ChainBase<3, 2, 1, 1> {
    static constexpr int NSIDE = 1;     // side[0] = r0 (read only by the dot product of the last level)
    double *p_new, *z1, *ap_new;
    const double *S;
    double beta, omega, d, calpha;
    FastDiv fd;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];
        omega = S[S_OMEGA];
        fd.set(d);
    }
    __device__ __forceinline__ void level0(bool out, size_t idx, const double (&raw)[3][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double pn = fma(beta, fma(-omega, raw[2][e], raw[1][e]), raw[0][e]);   // bicgstab.f90:176
            cc[0][e] = pn;
            u[e] = fd.div(pn);                                                           // chebyshev.f90:28-30
        }
        if (out) stg2(p_new + idx, cc[0][0], cc[0][1]);
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW, const double (&sd)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *acc) const {
        if (lv == 1) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                u[e] = fma(calpha, cin[0][e] - au[e], up[e]);                            // chebyshev.f90:35
                cout[0][e] = 0.0;
            }
            if (out) stg2(z1 + idx, u[0], u[1]);
        } else {
            u[0] = u[1] = 0.0;
            cout[0][0] = cout[0][1] = 0.0;
            if (out) {
                stg2(ap_new + idx, au[0], au[1]);
                acc[0] = fma(au[0], sd[0][0], acc[0]);                                   // :126 ap.r0
                acc[0] = fma(au[1], sd[0][1], acc[0]);
            }
        }
    }
};

// K2: s = r - alpha ap ; z2 = cbpr2(s) ; as = A z2 ; as.s, as.as
//     reads r,ap  writes s,z2,as  (40n B instead of 32n + 24n)
struct ChBiS : ChainBase<2, 2, 1, 2> {
    double *s, *z2, *as;
    const double *S;
    double alpha, d, calpha;
    FastDiv fd;
    __device__ __forceinline__ void init() { alpha = S[S_ALPHA]; fd.set(d); }
    __device__ __forceinline__ void level0(bool out, size_t idx, const double (&raw)[2][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double sv = fma(-alpha, raw[1][e], raw[0][e]);                         // bicgstab.f90:134
            cc[0][e] = sv;
            u[e] = fd.div(sv);
        }
        if (out) stg2(s + idx, cc[0][0], cc[0][1]);
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW, const double (&)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *acc) const {
        if (lv == 1) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                u[e] = fma(calpha, cin[0][e] - au[e], up[e]);
                cout[0][e] = cin[0][e];
            }
            if (out) stg2(z2 + idx, u[0], u[1]);
        } else {
            u[0] = u[1] = 0.0;
            cout[0][0] = cout[0][1] = 0.0;
            if (out) {
                stg2(as + idx, au[0], au[1]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    acc[0] = fma(au[e], cin[0][e], acc[0]);                              // :141 as.s
                    acc[1] = fma(au[e], au[e], acc[1]);                                  // :142 as.as
                }
            }
        }
    }
};

// K3: x += alpha z1 + omega z2 ; r = s - omega as ; acc0 = r.r ; acc1 = r.r0  (:148-152, :155, :161-164)
struct PBiUpdate : PwBase<2> {
    double *x, *r;
    const double *z1, *z2, *s, *as, *r0;
    const double *S;
    double alpha, omega;
    __device__ __forceinline__ void init() {
        alpha = S[S_ALPHA];
        omega = S[S_OMEGA];
    }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double vx[VEC], v1[VEC], v2[VEC], vs[VEC], va[VEC], v0[VEC], vr[VEC];
        KL_LD(VEC, v1, z1, i)
        KL_LD(VEC, v2, z2, i)
        KL_LD(VEC, vs, s, i)
        KL_LD(VEC, va, as, i)
        KL_LD(VEC, v0, r0, i)
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(x + i);
            vx[0] = t.x; vx[VEC - 1] = t.y;
        } else {
            vx[0] = x[i];
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            vx[v] = fma(omega, v2[v], fma(alpha, v1[v], vx[v]));
            vr[v] = fma(-omega, va[v], vs[v]);
            acc[0] = fma(vr[v], vr[v], acc[0]);
            acc[1] = fma(vr[v], v0[v], acc[1]);
        }
        KL_ST(VEC, x, i, vx)
        KL_ST(VEC, r, i, vr)
    }
};

// unfused direction update  p = r + beta (p - omega ap)  (:174-177), in place
struct PBiDir : PwBase<0> {
    double *p;
    const double *r, *ap;
    const double *S;
    double beta, omega;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];
        omega = S[S_OMEGA];
    }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *) const {
        double vr[VEC], va[VEC], vp[VEC];
        KL_LD(VEC, vr, r, i)
        KL_LD(VEC, va, ap, i)
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(p + i);
            vp[0] = t.x; vp[VEC - 1] = t.y;
        } else {
            vp[0] = p[i];
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) vp[v] = fma(beta, fma(-omega, va[v], vp[v]), vr[v]);
        KL_ST(VEC, p, i, vp)
    }
};


static int bicgstab_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                          double tol, int *iter, double *res_out, const kl_precond_t *M,
                          const double *params, int nparams) {
    if (!c || !A || !b || !x || !iter || !res_out) return KL_ERR_INVALID;
    KL_TRY(x0_check(c, b, x));
    Prob P;
    KL_TRY(prob_init(&P, c, A, M, params, nparams, nx, ny));
    const bool prec = P.pc.kind != KL_PC_NONE;
    const bool cb = P.pc.kind == KL_PC_CBPR2;
    const bool fused = c->opt_fuse && P.builtin_op() && (!prec || cb);
    const bool chain = fused && cb && chain_ok(&P, 2);   // cbpr2 and the operator in one pass (160n B/iteration)
    const size_t n = P.n;
    const int maxit = *iter;
    c->stats = kl_stats_t{};
    prof_reset(c);
    const cudaEvent_t evA = c->ev2, evB = c->ev3;     // owned by the handle (no leak on the error paths)
    KL_CUDA(c, cudaEventRecord(evA, c->stream));
    const bool dev = c->pointer_mode == KL_POINTER_DEVICE;
    KL_TRY(ws_reserve(c, 13 * ws_need(n)));
    ws_reset(c);
    double *r = ws_take<double>(c, n), *r0 = ws_take<double>(c, n);
    double *p0 = ws_take<double>(c, n), *p1 = ws_take<double>(c, n);
    double *ap0 = ws_take<double>(c, n), *ap1 = ws_take<double>(c, n);
    double *s = ws_take<double>(c, n), *as = ws_take<double>(c, n);
    double *dx = dev ? x : ws_take<double>(c, n);
    double *z1 = nullptr, *z2 = nullptr, *aux = nullptr, *aux2 = nullptr;
    if (prec) {
        z1 = ws_take<double>(c, n); z2 = ws_take<double>(c, n);
        aux = ws_take<double>(c, n); aux2 = ws_take<double>(c, n);
    }
    Cbpr2Coef cf{1.0, 0.0};
    if (cb) cf = cbpr2_coef(P.params);
    // x = 0 ; r = b ; r0 = r ; p = r0 (:114-118).  p_old = ap_old = 0 with beta = omega = 0
    // makes the first direction update produce p = r exactly.  KL_OPT_X0: x = x0 ; r = b - A x0.
    if (c->opt_x0) {
        KL_TRY(stage_in(c, dx, x, n));
        const double *db = b;
        if (!dev) {     // r0 is set from r below
            KL_TRY(stage_in(c, r0, b, n));
            db = r0;
        }
        KL_TRY(op_resid(&P, dx, db, r, false));
        double r_norm = 0.0;
        KL_TRY(x0_norm(c, r, n, &r_norm));
        if (r_norm < tol || r_norm == 0.0) {     // x0 already passes the test (r = 0 would make alpha 0/0)
            KL_TRY(x0_zero_step(c));
            *iter = 0;
            *res_out = r_norm;
            return KL_OK;
        }
    } else {
        KL_TRY(stage_in(c, r, b, n));
        KL_CUDA(c, cudaMemsetAsync(dx, 0, n * sizeof(double), c->stream));
    }
    KL_CUDA(c, cudaMemcpyAsync(r0, r, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    KL_CUDA(c, cudaMemsetAsync(p0, 0, n * sizeof(double), c->stream));
    KL_CUDA(c, cudaMemsetAsync(ap0, 0, n * sizeof(double), c->stream));
    KL_CUDA(c, cudaMemsetAsync(c->d_I, 0, sizeof(int) * I_COUNT, c->stream));
    {
        double S0[48] = {0};
        S0[S_TOL] = tol;
        KL_CUDA(c, cudaMemcpyAsync(c->d_S, S0, sizeof S0, cudaMemcpyHostToDevice, c->stream));
        int m1 = -1;
        KL_CUDA(c, cudaMemcpyAsync(c->d_I + I_CONV_AT, &m1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    {   // rr0 = r.r0
        PDot2 d;
        set_gate(d, c, false);
        d.a = r; d.b = r0; d.c = nullptr; d.d = nullptr;
        KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_RR, 0}));
    }
    KL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    double *pold = p0, *pnew = p1, *apold = ap0, *apnew = ap1;
    int done = 0, polls = 0, status = KL_NOT_CONVERGED;
    while (done < maxit) {
        int batch = c->opt_check_every;
        if (batch > maxit - done) batch = maxit - done;
        for (int k = 0; k < batch; ++k) {
            const double *zz1, *zz2;
            if (fused) {
                Halo H;
                const double *v3[3] = {r, pold, apold};
                if (chain) KL_TRY(halo_exchange_lines(&P, v3, 3, 2, &H));
                else KL_TRY(halo_exchange(&P, v3, 3, &H));
                if (cb && chain) {
                    ProfScope ps(c, 0, "bicg_dir_cbpr2_apply_dot (chain: p'=r+beta(p-omega ap); z1=cbpr2(p'); ap'=A z1; ap'.r0)", 56.0 * n);
                    ChBiDir f;
                    set_io(f, &P, v3, H);
                    set_gate(f, c, true);
                    f.p_new = pnew; f.z1 = z1; f.ap_new = apnew; f.side[0] = r0; f.S = c->d_S; f.d = cf.d; f.calpha = cf.alpha;
                    KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, PostBiAlpha{c->d_S}));
                    zz1 = z1;
                } else if (cb) {
                    FBiDir<true> f;
                    set_io(f, &P, v3, H);
                    set_gate(f, c, true);
                    f.p_new = pnew; f.out = z1; f.r0 = r0; f.S = c->d_S; f.d = cf.d; f.calpha = cf.alpha;
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, NoPost{}));
                    const double *v1[1] = {z1};
                    KL_TRY(halo_exchange(&P, v1, 1, &H));
                    FApplyDots g;
                    set_io(g, &P, v1, H);
                    set_gate(g, c, true);
                    g.y = apnew; g.e1 = r0; g.e2 = nullptr; g.self2 = 1;
                    KL_TRY(launch_stencil(c, &P.op, g, P.nx, P.nyl, PostBiAlpha{c->d_S}));
                    zz1 = z1;
                } else {
                    FBiDir<false> f;
                    set_io(f, &P, v3, H);
                    set_gate(f, c, true);
                    f.p_new = pnew; f.out = apnew; f.r0 = r0; f.S = c->d_S; f.d = 1.0; f.calpha = 0.0;
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostBiAlpha{c->d_S}));
                    zz1 = pnew;
                }
                const double *v2[2] = {r, apnew};
                if (chain) KL_TRY(halo_exchange_lines(&P, v2, 2, 2, &H));
                else KL_TRY(halo_exchange(&P, v2, 2, &H));
                if (cb && chain) {
                    ProfScope ps(c, 1, "bicg_s_cbpr2_apply_dots (chain: s=r-alpha ap'; z2=cbpr2(s); as=A z2; as.s; as.as)", 40.0 * n);
                    ChBiS f;
                    set_io(f, &P, v2, H);
                    set_gate(f, c, true);
                    f.s = s; f.z2 = z2; f.as = as; f.S = c->d_S; f.d = cf.d; f.calpha = cf.alpha;
                    KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, PostBiOmega{c->d_S}));
                    zz2 = z2;
                } else if (cb) {
                    FBiS<true> f;
                    set_io(f, &P, v2, H);
                    set_gate(f, c, true);
                    f.s = s; f.out = z2; f.S = c->d_S; f.d = cf.d; f.calpha = cf.alpha;
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, NoPost{}));
                    const double *v1[1] = {z2};
                    KL_TRY(halo_exchange(&P, v1, 1, &H));
                    FApplyDots g;
                    set_io(g, &P, v1, H);
                    set_gate(g, c, true);
                    g.y = as; g.e1 = s; g.e2 = nullptr; g.self2 = 1;
                    KL_TRY(launch_stencil(c, &P.op, g, P.nx, P.nyl, PostBiOmega{c->d_S}));
                    zz2 = z2;
                } else {
                    FBiS<false> f;
                    set_io(f, &P, v2, H);
                    set_gate(f, c, true);
                    f.s = s; f.out = as; f.S = c->d_S; f.d = 1.0; f.calpha = 0.0;
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostBiOmega{c->d_S}));
                    zz2 = s;
                }
            } else {
                // one kernel per reference loop; p is updated in place (pnew == pold buffers unused)
                pnew = pold; apnew = apold;
                PBiDir d;
                set_gate(d, c, true);
                d.p = pnew; d.r = r; d.ap = apold; d.S = c->d_S;
                KL_TRY(launch_pointwise(c, d, n, NoPost{}));
                if (prec) { KL_TRY(pc_apply(&P, pnew, z1, aux, aux2, 0, true, NoPost{})); zz1 = z1; }
                else zz1 = pnew;
                KL_TRY(op_apply(&P, zz1, apnew, true));
                PDot2 d1;
                set_gate(d1, c, true);
                d1.a = apnew; d1.b = r0; d1.c = nullptr; d1.d = nullptr;
                KL_TRY(launch_pointwise(c, d1, n, PostBiAlpha{c->d_S}));
                PAxpy sx;
                set_gate(sx, c, true);
                sx.a = r; sx.b = apnew; sx.y = s; sx.S = c->d_S; sx.s_idx = S_ALPHA; sx.sign = -1.0;
                KL_TRY(launch_pointwise(c, sx, n, NoPost{}));
                if (prec) { KL_TRY(pc_apply(&P, s, z2, aux, aux2, 0, true, NoPost{})); zz2 = z2; }
                else zz2 = s;
                KL_TRY(op_apply(&P, zz2, as, true));
                PDot2 d2;
                set_gate(d2, c, true);
                d2.a = as; d2.b = s; d2.c = as; d2.d = as;
                KL_TRY(launch_pointwise(c, d2, n, PostBiOmega{c->d_S}));
            }
            {
                ProfScope ps(c, 2, "bicg_update_xr_dots (pointwise: x+=alpha z1+omega z2; r=s-omega as; r.r; r.r0)",
                             (prec ? 64.0 : 56.0) * n);
                PBiUpdate u;
                set_gate(u, c, true);
                u.x = dx; u.r = r; u.z1 = zz1; u.z2 = zz2; u.s = s; u.as = as; u.r0 = r0; u.S = c->d_S;
                KL_TRY(launch_pointwise(c, u, n, PostBiEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap}));
            }
            if (fused) {
                std::swap(pold, pnew);
                if (!cb || chain) std::swap(apold, apnew);   // K1 reads ap and writes ap' in the same kernel
                else apold = apnew;   // cb: K1 reads ap while a later kernel writes it: same buffer is safe
            }
        }
        done += batch;
        KL_TRY(read_back(c));
        ++polls;
        if (c->h_pinned_i[I_CONV_AT] >= 0) {
            status = c->h_pinned_i[I_BREAKDOWN] ? KL_BREAKDOWN : KL_OK;
            break;
        }
    }
    KL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    KL_TRY(stage_out(c, x, dx, n));
    KL_TRY(fetch_history(c));
    KL_CUDA(c, cudaEventRecord(evB, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    prof_resolve(c);
    float ms = 0, ms_tot = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    cudaEventElapsedTime(&ms_tot, evA, evB);
    const int its = c->h_pinned_i[I_ITER];
    c->stats.iterations = its;
    c->stats.cycles = polls;
    c->stats.solve_ms = ms;
    c->stats.total_ms = ms_tot;
    c->stats.algorithmic_bytes = (double)its * (cb ? (chain ? 160.0 : 184.0) : 136.0) * (double)n;
    *res_out = c->h_pinned[S_RES];
    if (status == KL_OK) *iter = c->h_pinned_i[I_CONV_AT];
    return status;
}

}  // namespace kl

using namespace kl;

extern "C" {

int kl_bicgstab(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                double tol, int *iter, double *res) {
    return bicgstab_solve(h, A, b, x, nx, ny, tol, iter, res, nullptr, nullptr, 0);
}
int kl_pbicgstab(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                 double tol, int *iter, double *res, const kl_precond_t *M, const double *params,
                 int nparams) {
    return bicgstab_solve(h, A, b, x, nx, ny, tol, iter, res, M, params, nparams);
}
int kl_pbicgstab_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                     double tol, int *max_iter, double *res, const kl_precond_t *M, const double *params,
                     int nparams) {
    return bicgstab_solve(h, A, b, x, nx, ny, tol, max_iter, res, M, params, nparams);
}

}  // extern "C"
