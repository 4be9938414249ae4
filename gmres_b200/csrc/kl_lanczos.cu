// kl_lanczos.cu -- Lanczos spectral estimate for the Chebyshev preconditioner bounds.
//
// The reference only claims this feature (README.md:11); every driver hard-codes
// params = (8.2, 0.2) (tests/test_poisson_mf.f90:38).  Definition (shared with the
// CPU twin oracle/krylov_extras.c ko_lanczos): k-step symmetric Lanczos on A from
// v1 = b/||b||, b = A*1; the extreme eigenvalues of the tridiagonal T_k (bisection
// on the Sturm sequence) are returned.
//
// Per step: K1  w = A v ; alpha = v.w          (stencil + dot, 24n B)
//           K2  w -= alpha v + beta_prev v_prev ; ||w||^2     (32n B)
//           K3  v_next = w / beta                              (16n B)
#include <math.h>

#include <vector>

#include "kl_ops.cuh"

namespace kl {


struct PLanUpdate : PwBase<1> {
    double *w;
    const double *v, *vp;
    const double *S;
    int it;
    double al, bp;
    __device__ __forceinline__ void init() {
        al = S[S_LAN + it];
        bp = it > 0 ? S[S_LAN + kLanMax + it - 1] : 0.0;
    }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double vw[VEC], vv[VEC], vq[VEC];
        KL_LD(VEC, vv, v, i)
        KL_LD(VEC, vq, vp, i)
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(w + i);
            vw[0] = t.x; vw[VEC - 1] = t.y;
        } else {
            vw[0] = w[i];
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            vw[e] = fma(-bp, vq[e], fma(-al, vv[e], vw[e]));
            acc[0] = fma(vw[e], vw[e], acc[0]);
        }
        KL_ST(VEC, w, i, vw)
    }
};
struct PFill : PwBase<0> {
    double *y;
    double val;
    __device__ __forceinline__ void init() {}
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *) const {
        double v[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] = val;
        KL_ST(VEC, y, i, v)
    }
};

static int sturm_count(const double *a, const double *b, int k, double x) {
    int cnt = 0;
    double q = a[0] - x;
    if (q < 0) ++cnt;
    for (int i = 1; i < k; ++i) {
        double den = (q != 0.0) ? q : 1e-300;
        q = (a[i] - x) - b[i - 1] * b[i - 1] / den;
        if (q < 0) ++cnt;
    }
    return cnt;
}
static void tridiag_extremes(const double *a, const double *b, int k, double *lo_out, double *hi_out) {
    double lo = a[0], hi = a[0];
    for (int i = 0; i < k; ++i) {
        double rad = (i > 0 ? fabs(b[i - 1]) : 0.0) + (i < k - 1 ? fabs(b[i]) : 0.0);
        if (a[i] - rad < lo) lo = a[i] - rad;
        if (a[i] + rad > hi) hi = a[i] + rad;
    }
    for (int which = 0; which < 2; ++which) {
        double l = lo, h = hi;
        int target = which == 0 ? 1 : k;
        for (int it = 0; it < 200; ++it) {
            double mid = 0.5 * (l + h);
            if (mid == l || mid == h) break;
            if (sturm_count(a, b, k, mid) >= target) h = mid; else l = mid;
        }
        if (which == 0) *lo_out = 0.5 * (l + h); else *hi_out = 0.5 * (l + h);
    }
}

}  // namespace kl

using namespace kl;

extern "C" int kl_lanczos(kl_handle_t h, const kl_operator_t *A, int nx, int ny, int steps,
                          double *theta_min, double *theta_max) {
    if (!h || !A || !theta_min || !theta_max || steps < 1 || steps > kLanMax) return KL_ERR_INVALID;
    Ctx *c = h;
    Prob P;
    KL_TRY(prob_init(&P, c, A, nullptr, nullptr, 0, nx, ny));
    if (!P.symmetric())
        return c->fail(KL_ERR_UNSUPPORTED, "kl_lanczos needs a symmetric operator: for KL_OP_STENCIL5 use "
                                           "kl_stencil5_spectrum");
    const size_t n = P.n;
    KL_TRY(ws_reserve(c, 3 * ws_need(n)));
    ws_reset(c);
    double *v = ws_take<double>(c, n), *vp = ws_take<double>(c, n), *w = ws_take<double>(c, n);
    KL_CUDA(c, cudaMemsetAsync(c->d_I, 0, sizeof(int) * I_COUNT, c->stream));
    int m1 = -1;
    KL_CUDA(c, cudaMemcpyAsync(c->d_I + I_CONV_AT, &m1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    // b = A*1 ; v = b/||b|| ; v_prev = 0
    PFill one;
    set_gate(one, c, false);
    one.y = vp; one.val = 1.0;
    KL_TRY(launch_pointwise(c, one, n, NoPost{}));
    KL_TRY(op_apply(&P, vp, w, false));
    PDot2 d;
    set_gate(d, c, false);
    d.a = w; d.b = w; d.c = nullptr; d.d = nullptr;
    KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_NORM, 1}));
    PScale sc;
    set_gate(sc, c, false);
    sc.in = w; sc.out = v; sc.S = c->d_S; sc.s_idx = S_NORM;
    KL_TRY(launch_pointwise(c, sc, n, NoPost{}));
    KL_CUDA(c, cudaMemsetAsync(vp, 0, n * sizeof(double), c->stream));
    for (int i = 0; i < steps; ++i) {
        if (P.builtin_op()) {
            Halo H;
            const double *vecs[1] = {v};
            KL_TRY(halo_exchange(&P, vecs, 1, &H));
            FApplyDots f;
            set_io(f, &P, vecs, H);
            set_gate(f, c, true);
            f.y = w; f.e1 = v; f.e2 = nullptr; f.self2 = 1;
            KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostLanAlpha{c->d_S, i}));
        } else {
            KL_TRY(op_apply(&P, v, w, true));
            PDot2 dd;
            set_gate(dd, c, true);
            dd.a = v; dd.b = w; dd.c = nullptr; dd.d = nullptr;
            KL_TRY(launch_pointwise(c, dd, n, PostLanAlpha{c->d_S, i}));
        }
        PLanUpdate u;
        set_gate(u, c, true);
        u.w = w; u.v = v; u.vp = vp; u.S = c->d_S; u.it = i;
        KL_TRY(launch_pointwise(c, u, n, PostLanBeta{c->d_S, c->d_I, i}));
        // v_prev = v ; v = w / beta  (rotate buffers)
        PScale s2;
        set_gate(s2, c, true);
        s2.in = w; s2.out = vp; s2.S = c->d_S; s2.s_idx = S_NORM;
        KL_TRY(launch_pointwise(c, s2, n, NoPost{}));
        double *t = vp; vp = v; v = t;
    }
    std::vector<double> ab(2 * kLanMax);
    KL_CUDA(c, cudaMemcpyAsync(ab.data(), c->d_S + S_LAN, sizeof(double) * 2 * kLanMax, cudaMemcpyDeviceToHost, c->stream));
    KL_TRY(read_back(c));
    int k = c->h_pinned_i[I_ITER];
    if (k < 1) return c->fail(KL_BREAKDOWN, "lanczos: no step completed");
    tridiag_extremes(ab.data(), ab.data() + kLanMax, k, theta_min, theta_max);
    return KL_OK;
}
