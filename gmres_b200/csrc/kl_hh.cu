// kl_hh.cu -- restarted GMRES with Walker's Householder orthogonalisation.
//
// Reference: src/gmres_hh.f90  gmres_hh_omp :211-385 (no preconditioner, no
// in-cycle exit), gmres_hh_prec_omp :388-566 (left preconditioner, in-cycle
// `converged` flag), calculate_verr :568-593.
//
// Data layout: the unit reflectors P are n x (m+1) column-major (ld = ldv);
// reflector i is zero in rows < i.  H, g, cs, sn as in kl_gmres.cu.
//
// KL_HH_SEQUENTIAL (the reference's order): a reflector sweep v <- P_k ... P_i v
// is a chain of point-wise kernels, each applying the previous reflector (axpy)
// and accumulating the dot product with the next one in the same pass
// (32n B per reflector instead of 40n).  The serial O(n) block of the reference
// (:305-321) becomes: the last kernel of the sweep also reduces
// sum_{t>j+1} w_t^2, one warp builds H(:,j), the Householder pivot and the Givens
// update on the device, and one point-wise kernel writes the new reflector.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "kl_gmres.cuh"

namespace kl {


// v = e_j - 2 P_j (P_j . e_j) fused with the dot against the next reflector
// (gmres_hh.f90:257-283, first trip of the i-loop).
struct PHhInit : PwBase<1> {
    double *v;
    const double *pj, *pnext;
    long long j;
    double d0;
    __device__ __forceinline__ void init() { d0 = pj[j]; }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double p[VEC], a[VEC];
        KL_LD(VEC, p, pj, i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            double ej = ((long long)(i + e) == j) ? 1.0 : 0.0;
            a[e] = fma(-(2.0 * p[e]), d0, ej);
        }
        KL_ST(VEC, v, i, a)
        if (pnext) {
            double q[VEC];
            KL_LD(VEC, q, pnext, i)
#pragma unroll
            for (int e = 0; e < VEC; ++e) acc[0] = fma(a[e], q[e], acc[0]);
        }
    }
};

// w = [y(0..n_out-1); 0] fused with the dot against reflector n_out-1 (gmres_hh.f90:356-357)
struct PHhLoadY : PwBase<1> {
    double *w;
    const double *y, *pnext;
    long long n_out;
    __device__ __forceinline__ void init() {}
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double a[VEC], q[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) a[e] = ((long long)(i + e) < n_out) ? y[i + e] : 0.0;
        KL_ST(VEC, w, i, a)
        KL_LD(VEC, q, pnext, i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[0] = fma(a[e], q[e], acc[0]);
    }
};

// last trip of the second sweep: w -= 2 P_j (P_j.w) and S2 = sum_{t >= j+2} w_t^2
struct PHhLast : PwBase<1> {
    double *w;
    const double *vprev;
    const double *S;
    long long tail0;   // first index of the tail sum (j+2); < 0: x += w instead (cycle end)
    double *x;
    double hprev;
    __device__ __forceinline__ void init() { hprev = S[S_TMP0]; }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double a[VEC], p[VEC];
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(w + i);
            a[0] = t.x; a[VEC - 1] = t.y;
        } else {
            a[0] = w[i];
        }
        KL_LD(VEC, p, vprev, i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) a[e] = fma(-hprev, p[e], a[e]);
        if (x) {   // gmres_hh.f90:374-378  x = x + w
            double xv[VEC];
            if (VEC == 2) {
                double2 t = *reinterpret_cast<const double2 *>(x + i);
                xv[0] = t.x; xv[VEC - 1] = t.y;
            } else {
                xv[0] = x[i];
            }
#pragma unroll
            for (int e = 0; e < VEC; ++e) xv[e] = xv[e] + a[e];
            KL_ST(VEC, x, i, xv)
        } else {
            KL_ST(VEC, w, i, a)
#pragma unroll
            for (int e = 0; e < VEC; ++e)
                if ((long long)(i + e) >= tail0) acc[0] = fma(a[e], a[e], acc[0]);
        }
    }
};

// new reflector P_{j+1} = w' / ||w'|| with w'(0..j) = 0, w'(j+1) = pivot' (gmres_hh.f90:315-318)
struct PHhNewReflector : PwBase<0> {
    const double *w;
    double *p_out;
    const double *S;
    long long piv;   // index j+1 (0 for the first reflector of a cycle)
    double pv;
    FastDiv fd;
    __device__ __forceinline__ void init() {
        fd.set(S[S_NORM]);
        pv = S[S_TMP1];
    }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *) const {
        double a[VEC];
        KL_LD(VEC, a, w, i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            long long t = (long long)(i + e);
            a[e] = t < piv ? 0.0 : fd.div(t == piv ? pv : a[e]);
        }
        KL_ST(VEC, p_out, i, a)
    }
};

// serial block of the reference by ONE WARP (gmres_hh.f90:305-345 / :486-526)
__global__ void k_hh_step(const GmresDev G, const double *w, const int j, const int prec_variant, const long long n) {
    extern __shared__ double sm[];
    if (G.I[I_CONV_AT] >= 0) return;
    const int lane = threadIdx.x;
    double *sh = sm;
    double *Hj = G.H + (size_t)j * G.ldh;
    for (int i = lane; i <= j; i += 32) {   // :306 H(1:j,j) = w(1:j)
        double t = w[i];
        sh[i] = t;
        Hj[i] = t;
    }
    double hj1 = 0.0;
    if (lane == 0) {
        if ((long long)j + 1 < n) {                              // :307 if (j < n)
            const double S2 = G.S[S_RED];
            const double piv = w[j + 1];
            const double tmp = sqrt(fma(piv, piv, S2));          // :308 norm2(w(j+1:n))
            hj1 = (piv > 0.0) ? -tmp : tmp;                      // :309-313
            const double pv = piv - hj1;                         // :316
            G.S[S_TMP1] = pv;
            G.S[S_NORM] = sqrt(fma(pv, pv, S2));                 // :317 norm2(w)
        } else {                                                 // j = n (m = n): no reflector left, H(j+1,j) = 0 (:66-67)
            hj1 = 0.0;
            G.S[S_TMP1] = 0.0;
            G.S[S_NORM] = 1.0;
        }
    }
    hj1 = __shfl_sync(0xffffffffu, hj1, 0);
    __syncwarp();
    const int conv_before = G.I[I_CONV_AT];
    givens_update_warp(G, j, hj1, lane, sm, false);
    if (lane == 0 && !prec_variant) {
        // gmres_hh_omp: no in-cycle exit (:340-344 commented out)
        if (G.I[I_BREAKDOWN] == 0) G.I[I_CONV_AT] = conv_before;
    }
}

// first reflector of a cycle (gmres_hh.f90:250-253 / :433-436)
__global__ void k_hh_first(const GmresDev G, const double *w) {
    if (threadIdx.x != 0) return;
    const double ss = G.S[S_RED];
    const double w0 = w[0];
    const double beta = sqrt(ss);
    const double sg = copysign(beta, w0);
    G.g[0] = -sg;                                            // :251
    const double pv = sg + w0;                               // :252
    double S2 = ss - w0 * w0;
    if (S2 < 0.0) S2 = 0.0;
    G.S[S_TMP1] = pv;
    G.S[S_NORM] = sqrt(fma(pv, pv, S2));                     // :253 norm2(w)
}


// ===========================================================================
// KL_HH_BLOCKED: compact-WY form.  Q_j = P_0 ... P_j = I - Y T Y^T with Y = [p_0 .. p_j],
// T upper triangular, T(:,j+1) = -2 T (Y^T p_{j+1}), T(j+1,j+1) = 2.  Per Arnoldi step the
// reflector products become three tall-skinny passes over Y (24 n j bytes instead of 64 n j):
//   v_j = e_j - Y (T Y(j,:)^T)                       k_hh_apply_wy (src = e_j)
//   s   = Y^T w                                      k_ts_tma<false>
//   w  -= Y (T^T s) ; u = Y^T w ; tail ||w||^2       k_ts_tma<true>
// and the O(j^2) triangular products run on one warp.  Ytop holds the first m+1 rows of Y
// (reflector i is zero above row i), which is all the scalar part ever needs.
// ===========================================================================
struct HhWy {
    double *T;      // (m+1) x (m+1) column-major, ldt = m+1
    double *Ytop;   // (m+2) x (m+1) column-major, ldy = m+2
    double *tvec, *svec;
    int ldt, ldy;
};

// The O(j^2) triangular products use 8 warps: one warp per output element, lanes over the
// reduction index, shuffle reduction (the one-warp versions took ~10 us each at j ~ 90).
// tvec(0..j) = T(0..j,0..j) * Ytop(row j, 0..j)      (v_j ; also used by calculate_verr)
__global__ void __launch_bounds__(256) k_wy_pre(const GmresDev G, const HhWy W, const int j, const int gated) {
    if (gated && G.I[I_CONV_AT] >= 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int r = wid; r <= j; r += 8) {
        double t = 0.0;
        for (int c = r + lane; c <= j; c += 32) t = fma(W.T[(size_t)c * W.ldt + r], W.Ytop[(size_t)c * W.ldy + j], t);
        t = warp_sum(t);
        if (lane == 0) W.tvec[r] = t;
    }
}
// cycle end: svec = Ytop(0..k-1, 0..k-1)^T y ; tvec = T_k svec    (x += [y;0] - Y tvec)
__global__ void k_wy_xs(const GmresDev G, const HhWy W, const int k) {
    extern __shared__ double sm[];
    for (int c = threadIdx.x; c < k; c += 32) {
        double t = 0.0;
        for (int r = c; r < k; ++r) t = fma(W.Ytop[(size_t)c * W.ldy + r], G.y[r], t);
        sm[c] = t;
    }
    __syncwarp();
    for (int r = threadIdx.x; r < k; r += 32) {
        double t = 0.0;
        for (int c = r; c < k; ++c) t = fma(W.T[(size_t)c * W.ldt + r], sm[c], t);
        W.tvec[r] = t;
    }
}

// out = src - Y(:,0..nc-1) t ; src = e_row (mode 1) or [y(0..row-1); 0] (mode 2) ; dst: store or x += .
template <int VEC>
__global__ void __launch_bounds__(kTsThreads)
k_hh_apply_wy(const double *__restrict__ Y, const size_t ldv, const int nc, const double *__restrict__ t,
              const int src_mode, const long long row, const double *__restrict__ yv, double *dst,
              const int add_to_dst, const size_t n, const int *__restrict__ flags) {
    griddep_wait();
    griddep_launch();
    if (flags && flags[I_CONV_AT] >= 0) return;
    extern __shared__ double sh[];
    for (int c = threadIdx.x; c < nc; c += kTsThreads) sh[c] = t[c];
    __syncthreads();
    const size_t nchunk = n / VEC;
    for (size_t ch = (size_t)blockIdx.x * kTsThreads + threadIdx.x; ch < nchunk;
         ch += (size_t)gridDim.x * kTsThreads) {
        const size_t r = ch * VEC;
        double a[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const long long rr = (long long)(r + e);
            a[e] = src_mode == 1 ? (rr == row ? 1.0 : 0.0) : (rr < row ? yv[rr] : 0.0);
        }
        int c = 0;
        for (; c + 8 <= nc; c += 8) {
            double v[8][VEC];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double *col = Y + (size_t)(c + q) * ldv + r;
                if (VEC == 2) {
                    double2 tt = ldg2(col);
                    v[q][0] = tt.x; v[q][VEC - 1] = tt.y;
                } else {
                    v[q][0] = __ldg(col);
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double hq = -sh[c + q];
#pragma unroll
                for (int e = 0; e < VEC; ++e) a[e] = fma(hq, v[q][e], a[e]);
            }
        }
        for (; c < nc; ++c) {
            const double *col = Y + (size_t)c * ldv + r;
            const double hq = -sh[c];
            if (VEC == 2) {
                double2 tt = ldg2(col);
                a[0] = fma(hq, tt.x, a[0]);
                a[VEC - 1] = fma(hq, tt.y, a[VEC - 1]);
            } else {
                a[0] = fma(hq, __ldg(col), a[0]);
            }
        }
        if (add_to_dst) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) a[e] = dst[r + e] + a[e];
        }
        if (VEC == 2) stg2(dst + r, a[0], a[VEC - 1]);
        else dst[r] = a[0];
    }
}

// first reflector of a cycle in WY form: k_hh_first + T(0,0) = 2 + Ytop(:,0)
__global__ void k_hh_first_wy(const GmresDev G, const HhWy W, const double *w) {
    const int lane = threadIdx.x;
    double pv = 0.0, nw = 1.0;
    if (lane == 0) {
        const double ss = G.S[S_RED];
        const double w0 = w[0];
        const double beta = sqrt(ss);
        const double sg = copysign(beta, w0);
        G.g[0] = -sg;
        pv = sg + w0;
        double S2 = ss - w0 * w0;
        if (S2 < 0.0) S2 = 0.0;
        nw = sqrt(fma(pv, pv, S2));
        G.S[S_TMP1] = pv;
        G.S[S_NORM] = nw;
        W.T[0] = 2.0;
    }
    pv = __shfl_sync(0xffffffffu, pv, 0);
    nw = __shfl_sync(0xffffffffu, nw, 0);
    for (int r = lane; r <= G.m; r += 32) W.Ytop[r] = (r == 0 ? pv : w[r]) / nw;
    // k_wy_pre of step 0, folded in: tvec(0) = T(0,0) * Ytop(0,0)
    if (lane == 0) W.tvec[0] = 2.0 * (pv / nw);
}

// serial block of the reference in WY form: H(:,j), Householder pivot, new column of Ytop and of T
// (8 warps), then the Givens update by warp 0 (gmres_hh.f90:305-345).  u = Y^T w (u[0..j]) and the
// tail sum u[j+1].
constexpr int kHhStepThreads = 1024;     // 32 warps: the O(j^2) triangular products are latency-bound chains of
                                          // L2 loads, one output element per warp -- more warps, fewer rounds
__global__ void __launch_bounds__(kHhStepThreads)
k_hh_step_wy(const GmresDev G, const HhWy W, const double *w, const double *u, const int j, const int prec_variant) {
    extern __shared__ double sm[];     // 3*(m+2) for Givens + (m+2) for z
    griddep_wait();
    griddep_launch();
    if (G.I[I_CONV_AT] >= 0) return;
    constexpr int NW = kHhStepThreads / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double *sh = sm, *sz = sm + 3 * (G.m + 2);
    __shared__ double s_sc[3];
    double *Hj = G.H + (size_t)j * G.ldh;
    for (int i = threadIdx.x; i <= j; i += kHhStepThreads) {          // :306 H(1:j,j) = w(1:j)
        const double t = w[i];
        sh[i] = t;
        Hj[i] = t;
    }
    if (threadIdx.x == 0) {
        const double S2 = u[j + 1];
        const double piv = w[j + 1];
        const double tmp = sqrt(fma(piv, piv, S2));         // :308 norm2(w(j+1:n))
        const double hj1 = (piv > 0.0) ? -tmp : tmp;        // :309-313
        const double pv = piv - hj1;                        // :316
        const double nw = sqrt(fma(pv, pv, S2));            // :317 norm2(w)
        G.S[S_TMP1] = pv;
        G.S[S_NORM] = nw;
        s_sc[0] = hj1; s_sc[1] = pv; s_sc[2] = nw;
    }
    __syncthreads();
    const double hj1 = s_sc[0], pv = s_sc[1], nw = s_sc[2];
    // Ytop(:, j+1) = masked w / nw
    for (int r = threadIdx.x; r <= G.m; r += kHhStepThreads)
        W.Ytop[(size_t)(j + 1) * W.ldy + r] = r <= j ? 0.0 : ((r == j + 1 ? pv : w[r]) / nw);
    // z = Y^T p_{j+1} = (u - sum_{r<=j} Ytop(r,:) w_r - Ytop(j+1,:) hj1) / nw
    for (int c = wid; c <= j; c += NW) {
        double t = 0.0;
        for (int r = c + lane; r <= j; r += 32) t = fma(W.Ytop[(size_t)c * W.ldy + r], sh[r], t);
        t = warp_sum(t);
        if (lane == 0) sz[c] = ((u[c] - t) - W.Ytop[(size_t)c * W.ldy + j + 1] * hj1) / nw;
    }
    __syncthreads();
    // T(0..j, j+1) = -2 T z ; T(j+1,j+1) = 2
    for (int r = wid; r <= j; r += NW) {
        double t = 0.0;
        for (int c = r + lane; c <= j; c += 32) t = fma(W.T[(size_t)c * W.ldt + r], sz[c], t);
        t = warp_sum(t);
        if (lane == 0) W.T[(size_t)(j + 1) * W.ldt + r] = -2.0 * t;
    }
    if (threadIdx.x == 0) W.T[(size_t)(j + 1) * W.ldt + j + 1] = 2.0;
    // k_wy_pre of the NEXT step, folded in (one launch less on the critical path of every step):
    //   tvec(0..j+1) = T(0..j+1, 0..j+1) * Ytop(row j+1, 0..j+1)
    __syncthreads();
    if (j + 1 < G.m) {
        const int jn = j + 1;
        for (int r = wid; r <= jn; r += NW) {
            double t = 0.0;
            for (int c = r + lane; c <= jn; c += 32) t = fma(W.T[(size_t)c * W.ldt + r], W.Ytop[(size_t)c * W.ldy + jn], t);
            t = warp_sum(t);
            if (lane == 0) W.tvec[r] = t;
        }
    }
    if (wid != 0) return;
    const int conv_before = G.I[I_CONV_AT];
    givens_update_warp(G, j, hj1, lane, sm, false);
    if (lane == 0 && !prec_variant) {
        if (G.I[I_BREAKDOWN] == 0) G.I[I_CONV_AT] = conv_before;
    }
}

static int launch_apply_wy(Ctx *c, const double *Y, size_t ldv, int nc, const double *t, int src_mode, long long row,
                           const double *yv, double *dst, int add, size_t n, bool gated) {
    const int vec = (n % 2 == 0 && ldv % 2 == 0) ? 2 : 1;
    size_t b = (n / vec + kTsThreads - 1) / kTsThreads;
    if (b > (size_t)kNumSM * 8) b = (size_t)kNumSM * 8;
    const size_t smem = sizeof(double) * (nc + 8);
    const int *fl = gated ? c->d_I : nullptr;
    const int addi = add;
    if (vec == 2)
        KL_CUDA(c, launch_k(c, false, k_hh_apply_wy<2>, dim3((unsigned)b), dim3(kTsThreads), smem, Y, ldv, nc, t, src_mode,
                            row, yv, dst, addi, n, fl));
    else
        KL_CUDA(c, launch_k(c, false, k_hh_apply_wy<1>, dim3((unsigned)b), dim3(kTsThreads), smem, Y, ldv, nc, t, src_mode,
                            row, yv, dst, addi, n, fl));
    c->stats.kernel_launches++;
    return KL_OK;
}

struct HhRun {
    Ctx *c;
    Prob *P;
    GmresDev G;
    double *Pm;     // reflectors
    size_t ldv, n;
    double bytes;
};

// chain: v <- apply reflectors idx[0], idx[1], ... (in that order) to the vector already in `v`
// whose dot with P_{first} is already in S_TMP0 (doubled).  Each kernel applies one reflector and
// dots with the next.  The last one is returned to the caller (it has a special epilogue).
static int hh_chain(HhRun &R, double *v, int first, int last, int dir, bool gated) {
    // applies reflectors first, first+dir, ..., up to but NOT including `last`'s application:
    // i.e. kernels for i = first .. last-dir, each: axpy(P_i) + dot(P_{i+dir})
    Ctx *c = R.c;
    for (int i = first; i != last; i += dir) {
        PMgsStep s;
        set_gate(s, c, gated);
        s.w = v; s.S = c->d_S;
        s.vprev = R.Pm + (size_t)i * R.ldv;
        s.vcur = R.Pm + (size_t)(i + dir) * R.ldv;
        s.want_norm = 0;
        KL_TRY(launch_pointwise(c, s, R.n, PostHh{c->d_S}));
        R.bytes += 32.0 * R.n;
    }
    return KL_OK;
}

int gmres_hh_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny, int m,
                          double tol, double *final_err, double *v_err, int *n_out_p, int *stages_out_p,
                          const kl_precond_t *M, const double *params, int nparams, int prec_variant) {
    if (!c || !A || !b || !x || !final_err || !v_err || !n_out_p || !stages_out_p) return KL_ERR_INVALID;
    if (m < 1 || m + 1 > kMaxCols) return c->fail(KL_ERR_INVALID, "restart length m out of range");
    if (c->nranks > 1) return c->fail(KL_ERR_UNSUPPORTED, "Householder GMRES is single-GPU in this release");
    KL_TRY(x0_check(c, b, x));
    Prob P;
    KL_TRY(prob_init(&P, c, A, prec_variant == 1 ? M : nullptr, params, nparams, nx, ny));
    const bool prec = P.pc.kind != KL_PC_NONE;
    const size_t n = P.n;
    // j runs to m and the reference indexes v_j(j), so m <= n; m = n takes the `j < n` else-branch (gmres_hh.f90:53,66)
    if ((size_t)m > n) return c->fail(KL_ERR_INVALID, "m must not exceed the number of unknowns");
    const size_t ldv = (n + 31) & ~size_t(31);
    const int ldh = m + 1;
    c->stats = kl_stats_t{};
    prof_reset(c);
    const cudaEvent_t evA = c->ev2, evB = c->ev3;     // owned by the handle (no leak on the error paths)
    KL_CUDA(c, cudaEventRecord(evA, c->stream));
    const bool dev = c->pointer_mode == KL_POINTER_DEVICE;
    size_t need = ws_need(ldv * (size_t)(m + 1)) + (c->opt_verr ? ws_need(ldv * (size_t)m) : 0) + 7 * ws_need(n) +
                  ws_need((size_t)ldh * m) + 12 * ws_need(m + 2) + 3 * ws_need((size_t)(m + 2) * (m + 2));
    KL_TRY(ws_reserve(c, need));
    ws_reset(c);
    double *Pm = ws_take<double>(c, ldv * (size_t)(m + 1));
    double *Vb = c->opt_verr ? ws_take<double>(c, ldv * (size_t)m) : nullptr;
    double *w = ws_take<double>(c, n), *vj = ws_take<double>(c, n), *z = ws_take<double>(c, n);
    double *aux = ws_take<double>(c, n), *aux2 = ws_take<double>(c, n);
    double *db = dev ? const_cast<double *>(b) : ws_take<double>(c, n);
    double *dx = dev ? x : ws_take<double>(c, n);
    GmresDev G;
    G.H = ws_take<double>(c, (size_t)ldh * m);
    G.g = ws_take<double>(c, m + 2);
    G.cs = ws_take<double>(c, m + 2);
    G.sn = ws_take<double>(c, m + 2);
    G.y = ws_take<double>(c, m + 2);
    G.fe = ws_take<double>(c, m + 2);
    G.hvec = ws_take<double>(c, m + 2);
    G.hvec2 = G.hvec;
    double *d_gram = ws_take<double>(c, (size_t)(m + 2) * (m + 2));
    G.S = c->d_S; G.I = c->d_I; G.hist = c->d_hist; G.hist_cap = c->hist_cap;
    G.m = m; G.ldh = ldh; G.mf = (prec_variant == 2) ? 1 : 0;   // 2 = gmres_hh_dense: h_val < tol also stops (gmres_hh.f90:88)
    HhRun R{c, &P, G, Pm, ldv, n, 0.0};
    const bool blocked = c->opt_hh_mode == KL_HH_BLOCKED && ts_tma_ok(c, n, ldv, m);
    HhWy W;
    W.ldt = m + 1; W.ldy = m + 2;
    W.T = ws_take<double>(c, (size_t)(m + 1) * (m + 1));
    W.Ytop = ws_take<double>(c, (size_t)(m + 2) * (m + 1));
    W.tvec = ws_take<double>(c, m + 2);
    W.svec = ws_take<double>(c, m + 2);
    if (blocked) {
        KL_CUDA(c, cudaMemsetAsync(W.T, 0, sizeof(double) * (size_t)(m + 1) * (m + 1), c->stream));
        KL_CUDA(c, cudaMemsetAsync(W.Ytop, 0, sizeof(double) * (size_t)(m + 2) * (m + 1), c->stream));
    }

    if (!dev) KL_TRY(stage_in(c, db, b, n));
    if (c->opt_x0) KL_TRY(stage_in(c, dx, x, n));                               // x = x0 (KL_OPT_X0)
    else KL_CUDA(c, cudaMemsetAsync(dx, 0, n * sizeof(double), c->stream));
    KL_CUDA(c, cudaMemsetAsync(G.fe, 0, (m + 2) * sizeof(double), c->stream));
    KL_CUDA(c, cudaMemsetAsync(c->d_I, 0, sizeof(int) * I_COUNT, c->stream));
    {
        double S0[48] = {0};
        S0[S_TOL] = tol;
        KL_CUDA(c, cudaMemcpyAsync(c->d_S, S0, sizeof S0, cudaMemcpyHostToDevice, c->stream));
        int m1 = -1;
        KL_CUDA(c, cudaMemcpyAsync(c->d_I + I_CONV_AT, &m1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    {   // beta0 = norm2(b) (:237)
        PDot2 d;
        set_gate(d, c, false);
        d.a = db; d.b = db; d.c = nullptr; d.d = nullptr;
        KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_BETA0, 1}));
    }
    if (c->opt_x0) {
        // as in gmres_mgsr_solve: x0 whose ||M^-1 (b - A x0)|| / ||b|| already passes the test returns before a cycle
        KL_TRY(op_resid(&P, dx, db, z, false));
        if (prec) KL_TRY(pc_apply(&P, z, w, aux, aux2, 0, false, NoPost{}));
        double beta = 0.0;
        KL_TRY(x0_norm(c, prec ? w : z, n, &beta));
        if (beta == 0.0 || beta / c->h_pinned[S_BETA0] < tol) {
            KL_TRY(x0_zero_step(c));
            for (int i = 0; i < m; ++i) final_err[i] = 0.0;
            for (int i = 0; i <= m; ++i) v_err[i] = 0.0;
            *n_out_p = 0;
            *stages_out_p = 1;
            return KL_OK;
        }
    }
    KL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    const int max_stages = c->opt_max_restarts;
    int status = KL_NOT_CONVERGED, n_out = 0, stages_out = 0, cycles = 0;
    const size_t gsm = sizeof(double) * 3 * (m + 2);
    // The cycle up to the back substitution is a fixed launch sequence (the convergence test is a device-side gate):
    // captured once and replayed as a CUDA graph (KL_OPT_USE_GRAPH).  At 1024^2 (BASELINE config 2) a step is
    // 7 launches around ~250 us of work and the gaps between them were ~10 % of the step.
    auto enqueue_cycle = [&]() -> int {
        const PdlScope pdl_scope(c, true);               // programmatic dependent launch (single GPU by construction)
        // g = 0 ; H = 0 (:241).  P = 0 is implicit: every reflector is fully written before use.
        KL_CUDA(c, cudaMemsetAsync(G.H, 0, sizeof(double) * (size_t)ldh * m, c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.g, 0, sizeof(double) * (m + 2), c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.cs, 0, sizeof(double) * (m + 2), c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.sn, 0, sizeof(double) * (m + 2), c->stream));
        // w = b - A x [; w = M^-1 w] (:243-248 / :425-431)
        if (prec) {
            KL_TRY(op_resid(&P, dx, db, z, false));
            KL_TRY(pc_apply(&P, z, w, aux, aux2, 1, false, NoPost{}));
        } else {
            KL_TRY(op_resid(&P, dx, db, w, false));
            PDot2 d;
            set_gate(d, c, false);
            d.a = w; d.b = w; d.c = nullptr; d.d = nullptr;
            KL_TRY(launch_pointwise(c, d, n, NoPost{}));
        }
        if (blocked) k_hh_first_wy<<<1, 32, 0, c->stream>>>(G, W, w);
        else k_hh_first<<<1, 32, 0, c->stream>>>(G, w);           // :250-252
        {
            PHhNewReflector f;                                // :253 P(:,1) = w / norm2(w)
            set_gate(f, c, false);
            f.w = w; f.p_out = Pm; f.S = c->d_S; f.piv = 0;
            KL_TRY(launch_pointwise(c, f, n, NoPost{}));
        }
        c->stats.kernel_launches++;
        R.bytes += 56.0 * n;
        for (int j = 0; j < m; ++j) {
            if (blocked) {
                const int nc = j + 1;
                // v_j = e_j - Y (T Ytop(j,:)^T) ; tvec = T Ytop(j,:)^T comes from the previous step's scalar kernel
                KL_TRY(launch_apply_wy(c, Pm, ldv, nc, W.tvec, 1, j, nullptr, vj, 0, n, true));
                if (prec) {
                    KL_TRY(op_apply(&P, vj, z, true));
                    KL_TRY(pc_apply(&P, z, w, aux, aux2, 0, true, NoPost{}));
                } else {
                    KL_TRY(op_apply(&P, vj, w, true));
                }
                // s = Y^T w ; t = T^T s ; w -= Y t fused with u = Y^T w and the tail norm
                // (t = T^T s is computed by the last block of the projection kernel, kl_tallskinny_tma.cuh TsTail;
                // tvec was consumed by launch_apply_wy above and is refilled for the next step by k_hh_step_wy)
                KL_TRY(launch_ts_tma(c, false, Pm, ldv, m + 1, w, n, nc, nullptr, W.svec, G, j, 0, true, -1, W.T, W.tvec, W.ldt));
                KL_TRY(launch_ts_tma(c, true, Pm, ldv, m + 1, w, n, nc, W.tvec, G.hvec, G, j, 0, true, (long long)j + 2));
                KL_CUDA(c, launch_k(c, false, k_hh_step_wy, dim3(1), dim3(kHhStepThreads), sizeof(double) * 4 * (m + 2), G, W,
                                    (const double *)w, (const double *)G.hvec, j, prec_variant));
                c->stats.kernel_launches += 1;
                PHhNewReflector f;
                set_gate(f, c, true, j, 1);
                f.w = w; f.p_out = Pm + (size_t)(j + 1) * ldv; f.S = c->d_S; f.piv = (long long)j + 1;
                KL_TRY(launch_pointwise(c, f, n, NoPost{}));
                R.bytes += (24.0 * nc + 32.0 + 16.0 + (prec ? 32.0 : 16.0)) * n;
                continue;
            }
            // v = P_0 ... P_j e_j  (:257-283): reflectors applied in the order j, j-1, ..., 0
            {
                PHhInit f;
                set_gate(f, c, true);
                f.v = vj; f.pj = Pm + (size_t)j * ldv; f.pnext = j > 0 ? Pm + (size_t)(j - 1) * ldv : nullptr;
                f.j = j;
                KL_TRY(launch_pointwise(c, f, n, PostHh{c->d_S}));
                R.bytes += (j > 0 ? 24.0 : 16.0) * n;
            }
            if (j > 0) {
                KL_TRY(hh_chain(R, vj, j - 1, 0, -1, true));
                // last: apply P_0 (no further dot)
                PMgsStep s;
                set_gate(s, c, true);
                s.w = vj; s.S = c->d_S; s.vprev = Pm; s.vcur = nullptr; s.want_norm = 0;
                KL_TRY(launch_pointwise(c, s, n, NoPost{}));
                R.bytes += 24.0 * n;
            }
            // w = A v [; w = M^-1 w]  (:285 / :469-470)
            if (prec) {
                KL_TRY(op_apply(&P, vj, z, true));
                KL_TRY(pc_apply(&P, z, w, aux, aux2, 0, true, NoPost{}));
                R.bytes += 32.0 * n;
            } else {
                KL_TRY(op_apply(&P, vj, w, true));
                R.bytes += 16.0 * n;
            }
            // w = P_j ... P_0 w  (:290-304): order 0, 1, ..., j
            {
                PMgsStep s;   // dot with P_0 only
                set_gate(s, c, true);
                s.w = w; s.S = c->d_S; s.vprev = nullptr; s.vcur = Pm; s.want_norm = 0;
                KL_TRY(launch_pointwise(c, s, n, PostHh{c->d_S}));
                R.bytes += 16.0 * n;
            }
            KL_TRY(hh_chain(R, w, 0, j, +1, true));
            {
                PHhLast f;
                set_gate(f, c, true);
                f.w = w; f.vprev = Pm + (size_t)j * ldv; f.S = c->d_S; f.tail0 = (long long)j + 2; f.x = nullptr;
                KL_TRY(launch_pointwise(c, f, n, NoPost{}));
                R.bytes += 24.0 * n;
            }
            k_hh_step<<<1, 32, gsm, c->stream>>>(G, w, j, prec_variant, (long long)n);   // :305-345
            c->stats.kernel_launches++;
            {
                PHhNewReflector f;                                          // :315-318
                set_gate(f, c, true, j, 1);
                f.w = w; f.p_out = Pm + (size_t)(j + 1) * ldv; f.S = c->d_S; f.piv = (long long)j + 1;
                KL_TRY(launch_pointwise(c, f, n, NoPost{}));
                R.bytes += 16.0 * n;
            }
        }
        KL_TRY(launch_backsolve(c, G));                                    // :350-354
        return KL_OK;
    };
    const bool use_graph = c->opt_use_graph && !c->opt_profile && P.builtin_op() && c->opt_fuse &&
                           (P.pc.kind == KL_PC_NONE || P.pc.kind == KL_PC_CBPR2 || P.pc.kind == KL_PC_CHEB);
    GraphKey gk;
    if (use_graph) {
        gk.add('H').add(nx).add(ny).add(m).add(prec_variant).add(P.op.kind).add(P.op.eps_x).add(P.op.eps_y).add(P.w5)
            .add(P.pc.kind).add(P.pc.degree).add(P.params).add(c->opt_hh_mode).add(c->opt_tma).add(c->opt_chain)
            .add(c->opt_stencil_rows).add(c->opt_stencil_tail).add(c->opt_stencil_stagger).add(c->opt_verr).add(c->opt_pdl)
            .add(c->opt_reverse).add(c->opt_persistent)
            .add(c->ws).add(db).add(dx).add(Pm).add(G.H);
    }
    for (int k = 1; k <= max_stages; ++k) {
        ++cycles;
        Ctx::GraphEntry *ge = use_graph ? graph_find(c, gk.s) : nullptr;
        if (use_graph && !ge && k >= 2) {      // the first cycle of a handle's first solve runs eagerly
            const double b0 = R.bytes;
            const long long l0 = c->stats.kernel_launches;
            KL_TRY(graph_begin(c));
            const int rc = enqueue_cycle();
            if (rc < 0) {
                Ctx::GraphEntry *dummy = nullptr;
                graph_end(c, std::string(), 0.0, 0, &dummy);
                graph_clear(c);
                return rc;
            }
            KL_TRY(graph_end(c, gk.s, R.bytes - b0, c->stats.kernel_launches - l0, &ge));
            R.bytes = b0;
            c->stats.kernel_launches = l0;
        }
        if (ge) {
            KL_CUDA(c, cudaGraphLaunch(ge->exec, c->stream));
            R.bytes += ge->bytes;
            c->stats.kernel_launches += ge->launches;
        } else {
            KL_TRY(enqueue_cycle());
        }
        KL_TRY(read_back(c));
        n_out = c->h_pinned_i[I_NOUT];
        // w = [y;0] ; w = P_0 ... P_{n_out-1} w ; x += w  (:356-378)
        if (blocked) {
            k_wy_xs<<<1, 32, sizeof(double) * (m + 2), c->stream>>>(G, W, n_out);
            c->stats.kernel_launches++;
            KL_TRY(launch_apply_wy(c, Pm, ldv, n_out, W.tvec, 2, n_out, G.y, dx, 1, n, false));
            R.bytes += (8.0 * n_out + 16.0) * n;
        } else {
            PHhLoadY f;
            set_gate(f, c, false);
            f.w = w; f.y = G.y; f.pnext = Pm + (size_t)(n_out - 1) * ldv; f.n_out = n_out;
            KL_TRY(launch_pointwise(c, f, n, PostHh{c->d_S}));
            KL_TRY(hh_chain(R, w, n_out - 1, 0, -1, false));
            PHhLast g;
            set_gate(g, c, false);
            g.w = w; g.vprev = Pm; g.S = c->d_S; g.tail0 = -1; g.x = dx;
            KL_TRY(launch_pointwise(c, g, n, NoPost{}));
            R.bytes += (32.0 * n_out + 24.0) * n;
        }
        stages_out = k;                                                    // :381
        if (c->h_pinned_i[I_BREAKDOWN]) { status = KL_BREAKDOWN; break; }
        if (c->h_pinned[S_RES] < tol) { status = KL_OK; break; }           // :382
        if (prec_variant == 2 && c->h_pinned[S_HVAL] < tol) { status = KL_OK; break; }   // gmres_hh.f90:108 (dense)
    }
    KL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    KL_TRY(stage_out(c, x, dx, n));
    KL_CUDA(c, cudaMemcpyAsync(final_err, G.fe, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream));
    KL_TRY(fetch_history(c));
    for (int i = 0; i <= m; ++i) v_err[i] = 0.0;
    c->stats.orth_frobenius = NAN;
    if (c->opt_verr && n_out >= 1) {
        // calculate_verr (:568-593): V_i = P_0 ... P_i e_i, i < n_out
        for (int i = 0; i < n_out; ++i) {
            double *Vi = Vb + (size_t)i * ldv;
            if (blocked) {
                k_wy_pre<<<1, 256, 0, c->stream>>>(G, W, i, 0);
                KL_TRY(launch_apply_wy(c, Pm, ldv, i + 1, W.tvec, 1, i, nullptr, Vi, 0, n, false));
                continue;
            }
            PHhInit f;
            set_gate(f, c, false);
            f.v = Vi; f.pj = Pm + (size_t)i * ldv; f.pnext = i > 0 ? Pm + (size_t)(i - 1) * ldv : nullptr;
            f.j = i;
            KL_TRY(launch_pointwise(c, f, n, PostHh{c->d_S}));
            if (i > 0) {
                KL_TRY(hh_chain(R, Vi, i - 1, 0, -1, false));
                PMgsStep s;
                set_gate(s, c, false);
                s.w = Vi; s.S = c->d_S; s.vprev = Pm; s.vcur = nullptr; s.want_norm = 0;
                KL_TRY(launch_pointwise(c, s, n, NoPost{}));
            }
        }
        std::vector<double> gr;
        KL_TRY(gram_lower(c, Vb, ldv, n, n_out, d_gram, gr));
        double fro = 0.0;
        for (int col = 0; col < n_out; ++col)
            for (int i = 0; i <= col; ++i) {
                double d = gr[(size_t)col * n_out + i] - (i == col ? 1.0 : 0.0);
                fro += (i == col ? 1.0 : 2.0) * d * d;
            }
        c->stats.orth_frobenius = sqrt(fro);
        for (int i = 1; i < n_out; ++i)                                   // :587-591
            for (int jj = 0; jj < i; ++jj) {
                double d = gr[(size_t)i * n_out + jj];
                v_err[i] = v_err[i] + 2.0 * (d * d);
            }
    }
    KL_CUDA(c, cudaEventRecord(evB, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    float ms = 0, ms_tot = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    cudaEventElapsedTime(&ms_tot, evA, evB);
    c->stats.iterations = c->h_pinned_i[I_ITER];
    c->stats.cycles = cycles;
    c->stats.solve_ms = ms;
    c->stats.total_ms = ms_tot;
    c->stats.algorithmic_bytes = R.bytes;
    *n_out_p = n_out;
    *stages_out_p = stages_out;
    return status;
}

}  // namespace kl

using namespace kl;

extern "C" {

int kl_gmres_hh_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny, int m,
                    double tol, double *final_err, double *v_err, int *n_out, int *stages_out) {
    return gmres_hh_solve(h, A, b, x, nx, ny, m, tol, final_err, v_err, n_out, stages_out, nullptr, nullptr, 0, 0);
}
int kl_gmres_hh_prec_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                         int m, double tol, double *final_err, double *v_err, int *n_out, int *stages_out,
                         const kl_precond_t *M, const double *params, int nparams) {
    return gmres_hh_solve(h, A, b, x, nx, ny, m, tol, final_err, v_err, n_out, stages_out, M, params, nparams, 1);
}

}  // extern "C"
