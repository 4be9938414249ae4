// kl_posts.cuh -- "post" functors: the scalar recurrences that follow a reduction (alpha = rr / p.Ap, the Givens
// bookkeeping, ...).  They run in ONE thread of the LAST block of the reducing kernel (single GPU, or several GPUs
// with the in-kernel NVLink all-reduce) or in a one-thread kernel after the all-reduce.  The kernels are not
// templated on them: PostAny carries any of them by value and dispatches at run time (one call per kernel launch),
// which keeps the number of kernel instantiations at (functor x operator) instead of (functor x operator x post).
#pragma once

namespace kl {

constexpr int kLanMax = 256;    // Lanczos steps kept in the scalar block (S_LAN ..)

struct GmresDev {
    double *H;      // (m+1) x m, ldh = m+1
    double *g, *cs, *sn, *y, *fe, *hvec, *hvec2;
    double *S;
    int *I;
    double *hist;
    int hist_cap;
    int m, ldh;
    int mf;         // 1: gmres_mgsr_mf semantics (h_val < tol also stops; :172)
};

struct NoPost {
    __device__ __forceinline__ void run() const {}
};

struct PostStoreRed {   // S[dst] = S_RED[0]  (optionally sqrt)
    double *S;
    int dst;
    int do_sqrt;
    __device__ __forceinline__ void run() const {
        double v = S[S_RED];
        S[dst] = do_sqrt ? sqrt(v) : v;
    }
};

struct PostCgAlpha {  // cg.f90:124-126  alpha = rr / (ax.p)
    double *S;
    __device__ __forceinline__ void run() const {
        S[S_PAP] = S[S_RED];
        S[S_ALPHA] = S[S_RR] / S[S_RED];
    }
};

// end of a CG iteration: residual, history, convergence test (cg.f90:135-149)
__device__ __forceinline__ void cg_record(double *S, int *I, double *hist, int hist_cap, double res) {
    S[S_RES] = res;
    int it = I[I_ITER] + 1;
    I[I_ITER] = it;
    int hl = I[I_HIST];
    if (hl < hist_cap) hist[hl] = res;
    I[I_HIST] = hl + 1;
    if (res < S[S_TOL]) I[I_CONV_AT] = it;          // cg.f90:144-149
    else if (!(res == res)) { I[I_BREAKDOWN] = 1; I[I_CONV_AT] = it; }
}

struct PostCgEnd {
    double *S;
    int *I;
    double *hist;
    int hist_cap;
    int precond;  // 0: S_RED[0] = r.r (cg.f90:135-138) ; 1: S_RED[0] = r.z, r.r in S_TMP0 (cg.f90:219-226)
                  // 2: S_RED[0] = r.r, S_RED[1] = r.z (fused update + preconditioner kernel)
    __device__ __forceinline__ void run() const {
        double num = precond == 2 ? S[S_RED + 1] : S[S_RED];
        double rr2 = precond == 1 ? S[S_TMP0] : S[S_RED];
        S[S_BETA] = num / S[S_RR];
        S[S_RR] = num;
        cg_record(S, I, hist, hist_cap, sqrt(rr2));
    }
};

// One-pass CG (ChCg, kl_cg.cu).  S_RED = rho = r.r, gamma = p.Ap, sigma = r.Ap, delta = Ap.Ap of the iterate the
// pass produced.  alpha = rho / gamma is the reference's formula on true dot products (cg.f90:124-126).  beta needs
// ||r - alpha Ap||^2, the next pass's r.r; it is predicted by expanding the square, rho - 2 alpha sigma +
// alpha^2 delta, so that the next pass can form the direction in the same sweep.  The alpha and beta being replaced
// are kept in S_ALPHA_PREV / S_BETA_PREV: the second pass of a pair (ChCgPass<kCgPairB>) rebuilds the direction
// and the x update of the iteration before it.
__device__ __forceinline__ void cg_onepass_scalars(double *S) {
    const double rho = S[S_RED], gam = S[S_RED + 1], sig = S[S_RED + 2], del = S[S_RED + 3];
    const double alpha = rho / gam;
    S[S_ALPHA_PREV] = S[S_ALPHA];
    S[S_BETA_PREV] = S[S_BETA];
    S[S_PAP] = gam;
    S[S_ALPHA] = alpha;
    S[S_BETA] = (rho - 2.0 * alpha * sig + alpha * alpha * del) / rho;
    S[S_RR] = rho;
}
struct PostCgOnePassInit {   // after the prologue (sums of r_0 = p_0): alpha_0, beta_0
    double *S;
    __device__ __forceinline__ void run() const { cg_onepass_scalars(S); }
};
struct PostCgOnePass {       // after a pass: PostCgEnd's bookkeeping on the true ||r||, then alpha and beta
    double *S;
    int *I;
    double *hist;
    int hist_cap;
    __device__ __forceinline__ void run() const {
        cg_onepass_scalars(S);
        cg_record(S, I, hist, hist_cap, sqrt(S[S_RED]));
    }
};

struct PostBeta {   // gmres_mgsr.f90:322-323  beta = norm2(w) ; g(1) = beta
    GmresDev G;
    __device__ __forceinline__ void run() const {
        double beta = sqrt(G.S[S_RED]);
        G.S[S_NORM] = beta;
        G.g[0] = beta;
    }
};

struct PostMgs {
    GmresDev G;
    int j, i_cur;
    __device__ __forceinline__ void run() const {
        double h = G.S[S_RED];
        G.S[S_TMP0] = h;
        double *Hj = G.H + (size_t)j * G.ldh;
        Hj[i_cur] = Hj[i_cur] + h;
    }
};

struct PostHh {   // S_TMP0 = 2 * dot   (the "2.0d0*P*dot" factor of gmres_hh.f90:280)
    double *S;
    __device__ __forceinline__ void run() const { S[S_TMP0] = 2.0 * S[S_RED]; }
};

struct PostBiAlpha {   // :130 alpha = rr0 / ap_r0
    double *S;
    __device__ __forceinline__ void run() const { S[S_ALPHA] = S[S_RR] / S[S_RED]; }
};

struct PostBiOmega {   // :146 omega = as_s / as_as
    double *S;
    __device__ __forceinline__ void run() const { S[S_OMEGA] = S[S_RED] / S[S_RED + 1]; }
};

struct PostBiEnd {     // :154-173
    double *S;
    int *I;
    double *hist;
    int hist_cap;
    __device__ __forceinline__ void run() const {
        double res = sqrt(S[S_RED]);
        double r_r0_new = S[S_RED + 1];
        S[S_RES] = res;
        S[S_BETA] = (r_r0_new / S[S_RR]) * (S[S_ALPHA] / S[S_OMEGA]);
        S[S_RR] = r_r0_new;
        int it = I[I_ITER] + 1;
        I[I_ITER] = it;
        int hl = I[I_HIST];
        if (hl < hist_cap) hist[hl] = res;
        I[I_HIST] = hl + 1;
        if (res < S[S_TOL]) I[I_CONV_AT] = it;
        else if (!(res == res)) { I[I_BREAKDOWN] = 1; I[I_CONV_AT] = it; }
    }
};

struct PostLanAlpha {
    double *S;
    int step;
    __device__ __forceinline__ void run() const { S[S_LAN + step] = S[S_RED]; }
};

struct PostLanBeta {
    double *S;
    int *I;
    int step;
    __device__ __forceinline__ void run() const {
        double bt = sqrt(S[S_RED]);
        S[S_LAN + kLanMax + step] = bt;
        S[S_NORM] = bt;
        I[I_ITER] = step + 1;
        if (!(bt > 0.0)) I[I_CONV_AT] = step;
    }
};

enum PostKind { PK_NoPost, PK_PostStoreRed, PK_PostCgAlpha, PK_PostCgEnd, PK_PostCgOnePassInit, PK_PostCgOnePass, PK_PostBeta, PK_PostMgs, PK_PostHh, PK_PostBiAlpha, PK_PostBiOmega, PK_PostBiEnd, PK_PostLanAlpha, PK_PostLanBeta };
struct PostAny {
    int kind;
    union U {
        NoPost v_NoPost;
        PostStoreRed v_PostStoreRed;
        PostCgAlpha v_PostCgAlpha;
        PostCgEnd v_PostCgEnd;
        PostCgOnePassInit v_PostCgOnePassInit;
        PostCgOnePass v_PostCgOnePass;
        PostBeta v_PostBeta;
        PostMgs v_PostMgs;
        PostHh v_PostHh;
        PostBiAlpha v_PostBiAlpha;
        PostBiOmega v_PostBiOmega;
        PostBiEnd v_PostBiEnd;
        PostLanAlpha v_PostLanAlpha;
        PostLanBeta v_PostLanBeta;
    } u;
    // inlined into the reducing kernels' tails: a call would take the address of the kernel parameter and force a
    // copy of the whole union to local memory (216 B of stack and 12-16 more registers per kernel when it was
    // __noinline__); the switch is a few hundred bytes of code executed by one thread once per launch
    __device__ __forceinline__ void run() const {
        switch (kind) {
            case PK_NoPost: u.v_NoPost.run(); break;
            case PK_PostStoreRed: u.v_PostStoreRed.run(); break;
            case PK_PostCgAlpha: u.v_PostCgAlpha.run(); break;
            case PK_PostCgEnd: u.v_PostCgEnd.run(); break;
            case PK_PostCgOnePassInit: u.v_PostCgOnePassInit.run(); break;
            case PK_PostCgOnePass: u.v_PostCgOnePass.run(); break;
            case PK_PostBeta: u.v_PostBeta.run(); break;
            case PK_PostMgs: u.v_PostMgs.run(); break;
            case PK_PostHh: u.v_PostHh.run(); break;
            case PK_PostBiAlpha: u.v_PostBiAlpha.run(); break;
            case PK_PostBiOmega: u.v_PostBiOmega.run(); break;
            case PK_PostBiEnd: u.v_PostBiEnd.run(); break;
            case PK_PostLanAlpha: u.v_PostLanAlpha.run(); break;
            case PK_PostLanBeta: u.v_PostLanBeta.run(); break;
            default: break;
        }
    }
};
inline PostAny to_any(const NoPost &p) {
    PostAny a;
    a.kind = PK_NoPost;
    a.u.v_NoPost = p;
    return a;
}
inline PostAny to_any(const PostStoreRed &p) {
    PostAny a;
    a.kind = PK_PostStoreRed;
    a.u.v_PostStoreRed = p;
    return a;
}
inline PostAny to_any(const PostCgAlpha &p) {
    PostAny a;
    a.kind = PK_PostCgAlpha;
    a.u.v_PostCgAlpha = p;
    return a;
}
inline PostAny to_any(const PostCgEnd &p) {
    PostAny a;
    a.kind = PK_PostCgEnd;
    a.u.v_PostCgEnd = p;
    return a;
}
inline PostAny to_any(const PostCgOnePassInit &p) {
    PostAny a;
    a.kind = PK_PostCgOnePassInit;
    a.u.v_PostCgOnePassInit = p;
    return a;
}
inline PostAny to_any(const PostCgOnePass &p) {
    PostAny a;
    a.kind = PK_PostCgOnePass;
    a.u.v_PostCgOnePass = p;
    return a;
}
inline PostAny to_any(const PostBeta &p) {
    PostAny a;
    a.kind = PK_PostBeta;
    a.u.v_PostBeta = p;
    return a;
}
inline PostAny to_any(const PostMgs &p) {
    PostAny a;
    a.kind = PK_PostMgs;
    a.u.v_PostMgs = p;
    return a;
}
inline PostAny to_any(const PostHh &p) {
    PostAny a;
    a.kind = PK_PostHh;
    a.u.v_PostHh = p;
    return a;
}
inline PostAny to_any(const PostBiAlpha &p) {
    PostAny a;
    a.kind = PK_PostBiAlpha;
    a.u.v_PostBiAlpha = p;
    return a;
}
inline PostAny to_any(const PostBiOmega &p) {
    PostAny a;
    a.kind = PK_PostBiOmega;
    a.u.v_PostBiOmega = p;
    return a;
}
inline PostAny to_any(const PostBiEnd &p) {
    PostAny a;
    a.kind = PK_PostBiEnd;
    a.u.v_PostBiEnd = p;
    return a;
}
inline PostAny to_any(const PostLanAlpha &p) {
    PostAny a;
    a.kind = PK_PostLanAlpha;
    a.u.v_PostLanAlpha = p;
    return a;
}
inline PostAny to_any(const PostLanBeta &p) {
    PostAny a;
    a.kind = PK_PostLanBeta;
    a.u.v_PostLanBeta = p;
    return a;
}
inline PostAny to_any(const PostAny &p) { return p; }
template <class Post>
constexpr bool is_no_post() { return false; }
template <>
constexpr bool is_no_post<NoPost>() { return true; }

}  // namespace kl
