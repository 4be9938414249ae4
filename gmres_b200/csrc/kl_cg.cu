// kl_cg.cu -- Conjugate Gradient, plain and left-preconditioned.
//
// Reference: src/cg.f90  cg :11-42, pcg :44-81, cg_omp :83-152, pcg_omp :154-234.
// All four share one device implementation (the serial and OpenMP variants
// compute the same quantities; only their summation order differs).
//
// Plain CG, one GPU, from 2^27 unknowns on (default): 24n B per iteration, GROUPS of four temporally blocked passes
//   (16n + 16n + 16n + 48n, ChCgLook<J, STORE> below; r, p and x are stored every fourth iteration only).
// Plain CG, one GPU, 2^24 .. 2^27 unknowns (default): 36n B per iteration, PAIRS of temporally blocked passes
//   (24n + 48n, ChCgPass<kCgPairA / kCgPairB> below; p and x are stored every second iteration only).
// Plain CG, one GPU, 2^20 .. 2^24 unknowns (default): 48n B per iteration, ONE temporally blocked pass (ChCg below).
// Plain CG otherwise: 64n B per iteration, see FCgDirX2 / FCgRUpdate below (A applied twice, A p never stored).
// KL_OPT_CHAIN = 0 and PCG + cbpr2 -- per iteration 72n B for CG and 80n B for PCG + cbpr2:
//   K1  x += alpha_prev*p ; p' = z + beta*p ; ax = A p' ; ax.p'   reads z,p,x  writes p',ax,x   48n B
//   K2  r -= alpha ax ; r.r                                       reads r,ax   writes r         24n B
//       (pcg + cbpr2: r' = r - alpha ax ; z = cbpr2(r') ; r'.r' ; r'.z in one stencil pass     32n B)
// The x update of iteration k (cg.f90:127-129) is deferred into K1 of iteration k+1, which reads p anyway:
// the same fma on the same operands, so x is bit-identical to the reference order, and one read of p per
// iteration disappears (80n -> 72n).  The update still pending when the loop ends is flushed by one axpy.
// Generic path (user operator, KL_OPT_FUSE = 0, preconditioners other than cbpr2):
//   K1  p' = z + beta*p ; ax = A p' ; ax.p'         reads z,p   writes p',ax   32n B
//   K2  x += alpha p' ; r -= alpha ax ; r.r          reads x,p',r,ax writes x,r 48n B
//   K3  (pcg) z = M^-1 r ; r.z                       reads r     writes z       16n B
// alpha, beta, ||r||, the convergence flag and the residual history live on the
// device; the host polls once every KL_OPT_CHECK_EVERY iterations.
#include <math.h>

#include "kl_ops.cuh"

namespace kl {



// K1 with the deferred x update: x += alpha_prev * p_old ; p_new = z + beta*p_old ; ax = A p_new ; ax.p_new
// in[0] = z (r for plain CG), in[1] = p_old.  alpha_prev = S[S_ALPHA] of the previous iteration (0 before
// the first one, where p_old = 0 as well).
struct FCgDirX : StencilBase<2, 1> {
    double *p_new, *ax, *x;
    const double *S;
    double beta, alpha_prev;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];
        alpha_prev = S[S_ALPHA];
    }
    __device__ __forceinline__ double point(const double (&v)[2]) const { return fma(beta, v[1], v[0]); }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[2][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
        double vx[VEC];
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(x + idx);
            vx[0] = t.x; vx[VEC - 1] = t.y;
        } else {
            vx[0] = x[idx];
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            vx[v] = fma(alpha_prev, raw[1][v], vx[v]);        // cg.f90:128 of the previous iteration
            acc[0] = fma(au[v], cu[v], acc[0]);
        }
        KL_ST(VEC, x, idx, vx)
        KL_ST(VEC, p_new, idx, cu)
        KL_ST(VEC, ax, idx, au)
    }
};

// ---- plain CG with the operator applied twice instead of storing A p (64n B per iteration) ---------------
// K1: x += alpha_prev * p_old ; p_new = r + beta*p_old ; acc0 = (A p_new).p_new      reads r,p,x  writes p',x  40n
// K2: p_new = r + beta*p_old again (same fma => same bits) ; ax = A p_new ; r' = r - alpha ax ; acc0 = r'.r'
//                                                                                  reads r,p    writes r'    24n
// A p is never written to or read from HBM: five FP64 operations per point are cheaper than 16 bytes.  K2
// reuses the halo lines K1 exchanged (r and p_old have not changed), so there is no second exchange.
// Multi-GPU ("producer pushes", kCbPush in kl_internal.cuh): the CTAs that own the slab's first / last line also
// store that line of the NEW vector into the neighbour ranks' halo slots, so the next iteration needs no halo
// kernel; the all-reduce that ends the same kernel makes the lines visible before any consumer starts.
struct FCgDirX2 : StencilBase<2, 1> {
    static constexpr bool kPush = true;
    double *p_new, *x_new;     // x is ping-ponged like p and r: out-of-place streams reach a higher HBM efficiency
    const double *x;
    const double *S;
    double *push_first, *push_last;   // neighbours' slots for p_new's first / last line (nullptr: none)
    size_t last_off;                  // (ny_local - 1) * nx
    double beta, alpha_prev;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];
        alpha_prev = S[S_ALPHA];
    }
    __device__ __forceinline__ double point(const double (&v)[2]) const { return fma(beta, v[1], v[0]); }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[2][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc, int edge) const {
        double vx[VEC];
        KL_LD(VEC, vx, x, idx)
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            vx[v] = fma(alpha_prev, raw[1][v], vx[v]);        // cg.f90:128 of the previous iteration
            acc[0] = fma(au[v], cu[v], acc[0]);               // :118-122
        }
        KL_ST(VEC, x_new, idx, vx)
        KL_ST(VEC, p_new, idx, cu)
        if (edge) {
            if ((edge & 1) && push_first) { KL_ST(VEC, push_first, idx, cu) }
            if ((edge & 2) && push_last) { KL_ST(VEC, push_last, idx - last_off, cu) }
            __threadfence_system();
        }
    }
};
// kLateWait: under programmatic dependent launch K2 starts while K1 is still running.  Everything it touches
// before its first store() -- r, p_old, their halo lines, beta, the gate -- is older than K1; alpha (K1's last
// block) is read by late_init() after griddep_wait().
struct FCgRUpdate : StencilBase<2, 1> {
    static constexpr bool kPush = true;
    static constexpr bool kLateWait = true;
    static constexpr bool kReverse = true;     // starts on the lines of r and p that K1 read last (still in L2)
    double *r_new;
    const double *S;
    double *push_first, *push_last;   // neighbours' slots for r_new's first / last line
    size_t last_off;
    double beta, alpha;
    __device__ __forceinline__ void init() {
        beta = S[S_BETA];      // still the beta K1 used: PostCgEnd replaces it only after this kernel's last block
    }
    __device__ __forceinline__ void late_init() { alpha = S[S_ALPHA]; }
    __device__ __forceinline__ double point(const double (&v)[2]) const { return fma(beta, v[1], v[0]); }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[2][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc, int edge) const {
        double rn[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            rn[v] = fma(-alpha, au[v], raw[0][v]);            // cg.f90:130
            acc[0] = fma(rn[v], rn[v], acc[0]);               // :131-133
        }
        KL_ST(VEC, r_new, idx, rn)
        if (edge) {
            if ((edge & 1) && push_first) { KL_ST(VEC, push_first, idx, rn) }
            if ((edge & 2) && push_last) { KL_ST(VEC, push_last, idx - last_off, rn) }
            __threadfence_system();
        }
    }
};

// ---- plain CG in ONE pass per iteration (48n B, KL_OPT_CG_ONEPASS = 1) -------------------------------------
// A two-level temporally blocked chain (kl_chain_tma.cuh).  State at the start of pass k: r_k, p_k, x_k in HBM,
// alpha_k and beta_k in S[]:
//   level 0: u = p_k
//   level 1: A p_k ; r_{k+1} = r_k - alpha_k A p_k ; p_{k+1} = r_{k+1} + beta_k p_k       stores r_{k+1}, p_{k+1}
//   level 2: A p_{k+1} ; x_{k+1} = x_k + alpha_k p_k (x_k: side input, p_k re-read from the ring)   stores x_{k+1}
//            sums rho = r'.r', gamma = p'.Ap', sigma = r'.Ap', delta = Ap'.Ap'
// reads r, p, x and writes r', p', x'.  The point-wise operations are the two-kernel path's fmas on the same
// operands; only beta differs: PostCgOnePass predicts ||r_{k+2}||^2 from the sums of this pass instead of taking
// it from the next one (one reduction per iteration), see DESIGN.md section 3.2.
//
// ---- plain CG in PAIRS of passes (36n B per iteration, KL_OPT_CG_ONEPASS = 2) ------------------------------
// p_{k+1} = fma(beta_k, p_k, r_{k+1}) is one fma of two vectors that are in HBM anyway, and x feeds nothing in the
// recurrence.  So only every second pass stores p and x:
//   pass A (k -> k+1): the one-pass levels without the p and x stores           reads r_k, p_k        writes r_{k+1}
//   pass B (k+1 -> k+2): level 0 rebuilds u = p_{k+1} = fma(beta_k, p_k, r_{k+1}); level 1 as above with p_{k+1}
//     = u; level 2 rebuilds p_{k+1} at its output points and stores x_{k+2} = x_k + alpha_k p_k + alpha_{k+1} p_{k+1}
//     as the two fmas of two one-pass iterations              reads r_{k+1}, p_k, x_k   writes r_{k+2}, p_{k+2}, x_{k+2}
// 24n + 48n B per pair.  Every stored value and every sum is the one-pass path's fma chain on the same operands,
// and NIN, L (hence the CTA grid and the block-partial reduction order) are ChCg's: the results are bit-identical.
// Pass B takes alpha_k, beta_k from S_ALPHA_HIST / S_BETA_HIST (cg_onepass_scalars).
enum CgPass { kCgOne, kCgPairA, kCgPairB };
template <int MODE>
struct ChCgPass : ChainBase<2, 2, 1, 4> {
    static constexpr int NSIDE = MODE == kCgPairA ? 0 : 1;   // side[0] = x_k (read at the last level's output points)
    double *r_new, *p_new, *x_new;
    const double *S;
    double alpha, beta;
    double alpha0, beta0;     // pass B: alpha_k, beta_k of the pair's first iteration
    __device__ __forceinline__ void init() {
        alpha = S[S_ALPHA];
        beta = S[S_BETA];
        if (MODE == kCgPairB) {
            alpha0 = S[S_ALPHA_HIST];
            beta0 = S[S_BETA_HIST];
        }
    }
    __device__ __forceinline__ void level0(bool, size_t, const double (&raw)[2][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            u[e] = MODE == kCgPairB ? fma(beta0, raw[1][e], raw[0][e]) : raw[1][e];       // p_{k+1} : p_k
            cc[0][e] = 0.0;
        }
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW raw, const double (&sd)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *acc) const {
        if (lv == 1) {
            const double2 rv = raw(0), pv = raw(1);
            const double r2[2] = {rv.x, rv.y}, p2[2] = {pv.x, pv.y};
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                cout[0][e] = fma(-alpha, au[e], r2[e]);                                  // cg.f90:130
                u[e] = fma(beta, MODE == kCgPairB ? up[e] : p2[e], cout[0][e]);          // direction update
            }
            if (out) {
                stg2(r_new + idx, cout[0][0], cout[0][1]);
                if (MODE != kCgPairA) stg2(p_new + idx, u[0], u[1]);
            }
        } else {
            u[0] = u[1] = 0.0;
            cout[0][0] = cout[0][1] = 0.0;
            if (out) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    acc[0] = fma(cin[0][e], cin[0][e], acc[0]);                          // rho   = r'.r'
                    acc[1] = fma(au[e], up[e], acc[1]);                                  // gamma = p'.Ap'
                    acc[2] = fma(au[e], cin[0][e], acc[2]);                              // sigma = r'.Ap'
                    acc[3] = fma(au[e], au[e], acc[3]);                                  // delta = Ap'.Ap'
                }
                if (MODE != kCgPairA) {
                    const double2 pv = raw(1);
                    const double p2[2] = {pv.x, pv.y};
                    double xn[2];
                    if (MODE == kCgPairB) {
                        const double2 rv = raw(0);
                        const double r2[2] = {rv.x, rv.y};
#pragma unroll
                        for (int e = 0; e < 2; ++e)                                      // cg.f90:128, twice
                            xn[e] = fma(alpha, fma(beta0, p2[e], r2[e]), fma(alpha0, p2[e], sd[0][e]));
                    } else {
#pragma unroll
                        for (int e = 0; e < 2; ++e) xn[e] = fma(alpha, p2[e], sd[0][e]);    // cg.f90:128
                    }
                    stg2(x_new + idx, xn[0], xn[1]);
                }
            }
        }
    }
};
using ChCg = ChCgPass<kCgOne>;

// ---- plain CG in GROUPS of G passes (16n (G-1) + 48n B per G iterations, KL_OPT_CG_ONEPASS = 3) ------------------
// Recompute instead of store.  A group starts from r_k, p_k, x_k in HBM; its pass j = 1..G replays the j iterations
// k .. k+j-1 from them (J = j) and finds alpha_{k+j} and the predicted beta_{k+j} as the one-pass path does:
//   level 0:         u = p_k
//   level l = 1..J:  A p_{k+l-1} ; r_{k+l} = r_{k+l-1} - alpha_{k+l-1} A p_{k+l-1} ; p_{k+l} = r_{k+l} + beta_{k+l-1} p_{k+l-1}
//                    (r_k from the ring at level 1, then carried point-wise from level to level)
//                    STORE: x_{k+l} = x_k + alpha_k p_k + .. + alpha_{k+l-1} p_{k+l-1} (x_k from the ring at level 1,
//                    then carried), stored with r_{k+J} and p_{k+J} at level J
//   level J + 1:     A p_{k+J} ; rho, gamma, sigma, delta as ChCg's last level
// Passes 1..G-1 store nothing (reads r_k, p_k: 16n B); pass G stores (reads r_k, p_k, x_k, writes r, p, x: 48n B).
// Every point-wise value is the one-pass path's fma on the same operands.  The CTA grid is that of J + 1 levels, so
// the block-partial sums, hence alpha and beta, differ from the one-pass path's at rounding level.
// back = 0: the pass follows iteration k + J - 1, so alpha_{k+J-1} is S_ALPHA and the older ones are in the history;
// back = 1: the store pass that finishes a group after convergence at its pass J (one more iteration recorded).
template <int J, bool STORE>
struct ChCgLook : ChainBase<STORE ? 3 : 2, J + 1, STORE ? 2 : 1, 4> {
    static_assert(J >= 1 && J <= kCgHist + 1, "group depth");
    static constexpr bool SINGLE_GPU = true;
    // from three levels on: 2-line stages (a 12-line ring).  With 1-line stages the L retained lines leave only
    // 6 - L lines of lookahead, too few to cover the DRAM latency (measured at 16384^2 with G = 4: the 4-level store
    // pass took 2407 us against 2089 us for the 5-level one, which had 2-line stages)
    static constexpr int SR = J + 1 >= 3 ? 2 : 1;
    // store passes from four levels on: three 12-line inputs take 60-70 KB of ring, so at most 3 CTAs fit an SM
    // anyway; their register budget (168) then holds the four levels without spills (128 spilled 28-84 B)
    static constexpr int MINB = (STORE && J + 1 >= 4) ? 3 : ChainBase<STORE ? 3 : 2, J + 1, STORE ? 2 : 1, 4>::MINB;
    static constexpr int NC = STORE ? 2 : 1;
    double *r_new, *p_new, *x_new;
    const double *S;
    int back;
    double al[J], be[J];      // alpha_{k+l}, beta_{k+l}, l = 0..J-1
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int l = 0; l < J; ++l) {
            const int d = J - 1 - l + back;     // iterations before the current one
            al[l] = d == 0 ? S[S_ALPHA] : S[S_ALPHA_HIST + d - 1];
            be[l] = d == 0 ? S[S_BETA] : S[S_BETA_HIST + d - 1];
        }
    }
    __device__ __forceinline__ void level0(bool, size_t, const double (&raw)[STORE ? 3 : 2][2], double (&u)[2],
                                           double (&cc)[NC][2], double *) const {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            u[e] = raw[1][e];                                                            // p_k
#pragma unroll
            for (int k = 0; k < NC; ++k) cc[k][e] = 0.0;
        }
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[NC][2], RAW raw, const double (&)[1][2], double (&u)[2],
                                          double (&cout)[NC][2], double *acc) const {
        if (lv <= J) {
            double rk[2], xk[2];
            if (lv == 1) {
                const double2 rv = raw(0);
                rk[0] = rv.x; rk[1] = rv.y;
                if (STORE) {
                    const double2 xv = raw(STORE ? 2 : 0);
                    xk[0] = xv.x; xk[1] = xv.y;
                }
            } else {
                rk[0] = cin[0][0]; rk[1] = cin[0][1];
                xk[0] = cin[NC - 1][0]; xk[1] = cin[NC - 1][1];
            }
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                cout[0][e] = fma(-al[lv - 1], au[e], rk[e]);                             // cg.f90:130
                u[e] = fma(be[lv - 1], up[e], cout[0][e]);                               // direction update
                if (STORE) cout[NC - 1][e] = fma(al[lv - 1], up[e], xk[e]);              // cg.f90:128
            }
            if (STORE && lv == J && out) {
                stg2(r_new + idx, cout[0][0], cout[0][1]);
                stg2(p_new + idx, u[0], u[1]);
                stg2(x_new + idx, cout[NC - 1][0], cout[NC - 1][1]);
            }
        } else {
            u[0] = u[1] = 0.0;
#pragma unroll
            for (int k = 0; k < NC; ++k) cout[k][0] = cout[k][1] = 0.0;
            if (out) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    acc[0] = fma(cin[0][e], cin[0][e], acc[0]);                          // rho   = r'.r'
                    acc[1] = fma(au[e], up[e], acc[1]);                                  // gamma = p'.Ap'
                    acc[2] = fma(au[e], cin[0][e], acc[2]);                              // sigma = r'.Ap'
                    acc[3] = fma(au[e], au[e], acc[3]);                                  // delta = Ap'.Ap'
                }
            }
        }
    }
};
constexpr int kCgGroupMax = kCgHist + 1;

// Pass j of a group (store: also r, p, x), or the finishing store pass (back = 1, ungated, no post).  The names are
// the profile's (KL_OPT_PROFILE): classes 0..2 store nothing, 3..6 store at depth 1..4, 7 finishes a group.
static const char *const kCgLookName[2][kCgGroupMax] = {
    {"cg_group_look1 (chain, 2 levels: replay 1 iteration from r_k, p_k; A p; 4 dots; stores nothing)",
     "cg_group_look2 (chain, 3 levels: replay 2 iterations from r_k, p_k; A p; 4 dots; stores nothing)",
     "cg_group_look3 (chain, 4 levels: replay 3 iterations from r_k, p_k; A p; 4 dots; stores nothing)",
     nullptr},
    {"cg_group_store1 (chain, 2 levels: replay 1 iteration from r_k, p_k, x_k; store r, p, x; A p; 4 dots)",
     "cg_group_store2 (chain, 3 levels: replay 2 iterations from r_k, p_k, x_k; store r, p, x; A p; 4 dots)",
     "cg_group_store3 (chain, 4 levels: replay 3 iterations from r_k, p_k, x_k; store r, p, x; A p; 4 dots)",
     "cg_group_store4 (chain, 5 levels: replay 4 iterations from r_k, p_k, x_k; store r, p, x; A p; 4 dots)"}};
static const char kCgFinishName[] = "cg_group_finish (chain: x after convergence inside a group)";

template <int J, bool STORE>
static int cg_look_launch(Ctx *c, Prob *P, const double *r, const double *p, const double *x, double *r_new,
                          double *p_new, double *x_new, int back, bool gated) {
    Halo H{};
    const double *vecs[3] = {r, p, x};
    ChCgLook<J, STORE> f;
    set_io(f, P, vecs, H);
    set_gate(f, c, gated);
    f.r_new = r_new; f.p_new = p_new; f.x_new = x_new; f.S = c->d_S; f.back = back;
    if (back) return launch_chain(c, &P->op, f, P->nx, P->nyl, NoPost{});
    return launch_chain(c, &P->op, f, P->nx, P->nyl, PostCgOnePass{c->d_S, c->d_I, c->d_hist, c->hist_cap});
}
static int cg_look(Ctx *c, Prob *P, int J, bool store, const double *r, const double *p, const double *x,
                   double *r_new, double *p_new, double *x_new, int back, bool gated) {
#define KL_LOOK(JJ, ST) \
    if (J == JJ && store == ST) return cg_look_launch<JJ, ST>(c, P, r, p, x, r_new, p_new, x_new, back, gated);
    KL_LOOK(1, false) KL_LOOK(2, false) KL_LOOK(3, false)
    KL_LOOK(1, true) KL_LOOK(2, true) KL_LOOK(3, true) KL_LOOK(4, true)
#undef KL_LOOK
    return c->fail(KL_ERR_INVALID, "cg_look: group depth");
}

// Prologue of the one-pass path: the four sums of ChCg's last level for p_0 = r_0 (= b), no store.
struct FCgOnePassInit : StencilBase<1, 4> {
    __device__ __forceinline__ void init() {}
    __device__ __forceinline__ double point(const double (&v)[1]) const { return v[0]; }
    template <int VEC>
    __device__ __forceinline__ void store(size_t, const double (&)[1][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            acc[0] = fma(cu[v], cu[v], acc[0]);
            acc[1] = fma(au[v], cu[v], acc[1]);
            acc[2] = fma(au[v], cu[v], acc[2]);
            acc[3] = fma(au[v], au[v], acc[3]);
        }
    }
};

// K2 without x: r -= alpha ax ; acc0 = sum r*r     (cg.f90:130-133)
struct PCgUpdateR : PwBase<1> {
    double *r;
    const double *ax;
    const double *S;
    double alpha;
    __device__ __forceinline__ void init() { alpha = S[S_ALPHA]; }
    template <int VEC>
    __device__ __forceinline__ void elem(size_t i, double *acc) const {
        double vr[VEC], va[VEC];
        KL_LD(VEC, va, ax, i)
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(r + i);
            vr[0] = t.x; vr[VEC - 1] = t.y;
        } else {
            vr[0] = r[i];
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            vr[v] = fma(-alpha, va[v], vr[v]);
            acc[0] = fma(vr[v], vr[v], acc[0]);
        }
        KL_ST(VEC, r, i, vr)
    }
};

// PCG + cbpr2 without x: r' = r - alpha ax ; z = cbpr2(r') ; r'.r' ; r'.z   (cg.f90:209-218)
struct FPcgUpdateR : StencilBase<2, 2> {
    double *r_new, *z;
    const double *S;
    double alpha, d, calpha;
    FastDiv fd;
    __device__ __forceinline__ void init() {
        alpha = S[S_ALPHA];
        fd.set(d);
    }
    __device__ __forceinline__ double point(const double (&v)[2]) const { return fd.div(fma(-alpha, v[1], v[0])); }
    template <int VEC>
    __device__ __forceinline__ void store(size_t idx, const double (&raw)[2][VEC], const double (&cu)[VEC],
                                          const double (&au)[VEC], double *acc) const {
        double rn[VEC], zz[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            rn[v] = fma(-alpha, raw[1][v], raw[0][v]);        // :209
            zz[v] = fma(calpha, rn[v] - au[v], cu[v]);        // chebyshev.f90:35
            acc[0] = fma(rn[v], rn[v], acc[0]);               // :210
            acc[1] = fma(rn[v], zz[v], acc[1]);               // :216
        }
        KL_ST(VEC, r_new, idx, rn)
        KL_ST(VEC, z, idx, zz)
    }
};

// KL_OPT_CG_ONEPASS = -1: the one-pass path from this many unknowns on.  It won at every size of the sweep, 1.33x at
// 1024^2 .. 1.79x at 2048^2 (scripts/cg_onepass_sweep.py, profiles/r03_cg_onepass_sweep.json); the grids below 1 Mi
// unknowns (vectors resident in L2, not swept) keep the two-kernel iteration.
constexpr size_t kCgOnePassMin = (size_t)1 << 20;
// ... and pairs of passes (36n B per iteration) from this many on (scripts/cg_pair_sweep.py,
// profiles/r04_cg_pair_sweep.json).
constexpr size_t kCgPairMin = (size_t)1 << 24;
// ... and groups of passes from this many on (scripts/cg_group_sweep.py, profiles/r08_cg_group_sweep.json)
constexpr size_t kCgGroupMin = (size_t)1 << 27;

static int cg_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                    double tol, int *iter, double *res_out, const kl_precond_t *M, const double *params,
                    int nparams) {
    if (!c || !A || !b || !x || !iter || !res_out) return KL_ERR_INVALID;
    KL_TRY(x0_check(c, b, x));
    Prob P;
    KL_TRY(prob_init(&P, c, A, M, params, nparams, nx, ny));
    if (!P.symmetric())
        return c->fail(KL_ERR_UNSUPPORTED, "CG / PCG need a symmetric operator: KL_OP_STENCIL5 with wl != wr or wd != wu "
                                           "takes GMRES or BiCGSTAB");
    const bool prec = P.pc.kind != KL_PC_NONE;
    const bool fused = c->opt_fuse && P.builtin_op();
    const size_t n = P.n;
    const int maxit = *iter;
    c->stats = kl_stats_t{};
    prof_reset(c);
    const cudaEvent_t evA = c->ev2, evB = c->ev3;     // owned by the handle (no leak on the error paths)
    KL_CUDA(c, cudaEventRecord(evA, c->stream));

    const bool dev = c->pointer_mode == KL_POINTER_DEVICE;
    const bool fuse_pc = fused && P.pc.kind == KL_PC_CBPR2;   // update + cbpr2 in one pass
    const bool defer_x = fused && (!prec || fuse_pc);         // x update folded into the next K1 (72n / 80n B)
    const bool twice = defer_x && !prec && c->opt_chain;       // plain CG: apply A twice, never store A p (64n B)
    // plain CG in one chain pass per iteration (48n B) or in pairs of passes (36n B): single GPU (the chain needs a
    // two-line halo, which the multi-GPU producer-push protocol does not deliver)
    // groups of G passes need G + 1 levels
    const int G = c->opt_cg_group;
    int cg_pass = !(twice && c->nranks == 1 && chain_ok(&P, 2)) ? 0
                  : c->opt_cg_onepass >= 0 ? c->opt_cg_onepass
                  : (n >= kCgGroupMin ? 3 : (n >= kCgPairMin ? 2 : (n >= kCgOnePassMin ? 1 : 0)));
    if (cg_pass == 3 && !chain_ok(&P, G + 1)) cg_pass = 2;
    const bool onepass = cg_pass == 1, pair = cg_pass == 2, group = cg_pass == 3;
    const int nvec = 4 + (dev ? 0 : 1) + (prec ? 3 : 0) + ((fuse_pc || twice) ? 1 : 0) + (twice ? 1 : 0);
    KL_TRY(ws_reserve(c, nvec * ws_need(n)));
    ws_reset(c);
    double *r = ws_take<double>(c, n), *p0 = ws_take<double>(c, n), *p1 = ws_take<double>(c, n);
    double *ax = ws_take<double>(c, n);
    double *dx = dev ? x : ws_take<double>(c, n);
    double *z = r, *aux = nullptr, *aux2 = nullptr;
    double *r_alt = (fuse_pc || twice) ? ws_take<double>(c, n) : nullptr;
    double *x_cur = dx, *x_alt = twice ? ws_take<double>(c, n) : nullptr;
    // one-pass: x is ping-ponged from the first iteration on; start it where an odd / even maxit ends in dx
    // pairs: x moves once per pair; start it where maxit / 2 pairs end in dx (an odd maxit ends in a flush to dx)
    // groups: x moves once per group; start it where the ceil(maxit / G) store passes end in dx
    if ((onepass && (maxit & 1)) || (pair && ((maxit / 2) & 1)) || (group && (((maxit + G - 1) / G) & 1)))
        std::swap(x_cur, x_alt);
    double *const x_start = x_cur, *const x_other = x_alt;
    double *const r_start = r, *const r_other = r_alt;
    const Cbpr2Coef cf = fuse_pc ? cbpr2_coef(P.params) : Cbpr2Coef{1.0, 0.0};
    if (prec) {
        z = ws_take<double>(c, n);
        aux = ws_take<double>(c, n);
        aux2 = ws_take<double>(c, n);
    }
    // x0 = 0 ; r0 = b ; p0 = r0 (cg.f90:102-108).  KL_OPT_X0: r0 = b - A x0 with x0 in the buffer the iterations
    // start from (the two-kernel paths' first x update adds alpha = 0 times p = 0 to it, which leaves it as it is)
    if (c->opt_x0) {
        KL_TRY(stage_in(c, dx, x, n));
        const double *db = b;
        if (!dev) {     // ax is not read before the first iteration writes it
            KL_TRY(stage_in(c, ax, b, n));
            db = ax;
        }
        KL_TRY(op_resid(&P, dx, db, r, false));
        if (x_cur != dx) KL_CUDA(c, cudaMemcpyAsync(x_cur, dx, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        double r0_norm = 0.0;
        KL_TRY(x0_norm(c, r, n, &r0_norm));
        if (r0_norm < tol || r0_norm == 0.0) {     // x0 already passes the test (r0 = 0 would make alpha 0/0)
            KL_TRY(x0_zero_step(c));
            *iter = 0;
            *res_out = r0_norm;
            return KL_OK;
        }
    } else {
        KL_TRY(stage_in(c, r, b, n));
        KL_CUDA(c, cudaMemsetAsync(x_cur, 0, n * sizeof(double), c->stream));
    }
    // pairs: p_0 = r_0 gets a buffer of its own, as pass B of the first pair overwrites r_0's with r_2 (groups: so
    // that r and p ping-pong alike from the first group on)
    if (pair || group) KL_CUDA(c, cudaMemcpyAsync(p0, r, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    else KL_CUDA(c, cudaMemsetAsync(p0, 0, n * sizeof(double), c->stream));
    KL_CUDA(c, cudaMemsetAsync(c->d_I, 0, sizeof(int) * I_COUNT, c->stream));
    {
        double S0[32] = {0};
        S0[S_TOL] = tol;
        KL_CUDA(c, cudaMemcpyAsync(c->d_S, S0, sizeof S0, cudaMemcpyHostToDevice, c->stream));
        int m1 = -1;
        KL_CUDA(c, cudaMemcpyAsync(c->d_I + I_CONV_AT, &m1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    // multi-GPU, peer memory: the producing kernels push their boundary lines (slot 0 = r, slot 1 = p, parity =
    // iteration & 1); the lines of r0 = b and p0 = 0 are pushed here, the all-reduce of the dot product below is
    // the barrier that orders them before the first K1 on every rank
    const bool push = twice && comm_push_ok(c, P.nx) && c->opt_tma && P.nx >= 64;
    if (push) {
        const double *first[2] = {r, nullptr}, *last[2] = {r + (size_t)(P.nyl - 1) * P.nx, nullptr};
        const int slots[2] = {0, 1};
        KL_TRY(comm_push_lines(c, 2, first, last, slots, 0, P.nx));
    }
    // rr = r.z  (z = M^-1 r for pcg, cg.f90:182 ; z = r otherwise)
    // one-pass: rr, p.Ap, r.Ap and Ap.Ap for p_0 = r_0, then alpha_0 and the predicted beta_0
    if (prec) {
        KL_TRY(pc_apply(&P, r, z, aux, aux2, 2, false, PostStoreRed{c->d_S, S_RR, 0}));
    } else if (onepass || pair || group) {
        Halo H{};
        const double *vecs[1] = {r};
        FCgOnePassInit d;
        set_io(d, &P, vecs, H);
        set_gate(d, c, false);
        KL_TRY(launch_stencil(c, &P.op, d, P.nx, P.nyl, PostCgOnePassInit{c->d_S}));
    } else {
        PDot2 d;
        set_gate(d, c, false);
        d.a = r; d.b = r; d.c = nullptr; d.d = nullptr;
        KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_RR, 0}));
    }
    // S_BETA = 0 with p_old = 0 makes the first K1 produce p = z exactly.

    KL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    double *pold = p0, *pnew = p1;
    int done = 0, polls = 0;
    int status = KL_NOT_CONVERGED;
    // `count` iterations starting after iteration `done0`.  The buffer roles (r / r_alt, x_cur / x_alt, p_old / p_new)
    // alternate with period two, so an even batch leaves them as it found them and can be replayed as a CUDA graph.
    auto enqueue_iterations = [&](const int done0, const int batch) -> int {
        const int done = done0;
        for (int k = 0; k < batch; ++k) {
            if (group) {
                // pass j of its group replays j iterations from the group's r_k, p_k (x_k); the last pass of a group,
                // and of a group truncated by maxit, stores r, p and x, which then move to the other buffers
                const int it = done + k, j = it % G + 1;
                const bool store = j == G || it + 1 == maxit;
                ProfScope ps(c, store ? 2 + j : j - 1, kCgLookName[store][j - 1], (store ? 48.0 : 16.0) * n);
                KL_TRY(cg_look(c, &P, j, store, r, pold, x_cur, r_alt, pnew, x_alt, 0, true));
                if (store) {
                    std::swap(r, r_alt);
                    std::swap(x_cur, x_alt);
                    std::swap(pold, pnew);
                }
                z = r;
                continue;
            }
            if (pair && ((done + k) & 1) == 0) {
                // pass A: p_0 is in p0 from the prologue on, p alternates between p1 (written by the first pair) and p0
                ProfScope ps(c, 0, "cg_pair_a (chain: r-=alpha*A p; p=r+beta*p; A p; 4 dots)", 24.0 * n);
                Halo H{};
                const double *vecs[2] = {r, pold};
                ChCgPass<kCgPairA> f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.r_new = r_alt; f.p_new = nullptr; f.x_new = nullptr; f.S = c->d_S;
                KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, PostCgOnePass{c->d_S, c->d_I, c->d_hist, c->hist_cap}));
                std::swap(r, r_alt);
                z = r;
                continue;
            }
            if (pair) {
                ProfScope ps(c, 1, "cg_pair_b (chain: p=r+beta0*p0; r-=alpha*A p; p=r+beta*p; x+=alpha0*p0+alpha*p; A p; 4 dots)",
                             48.0 * n);
                Halo H{};
                const double *vecs[2] = {r, pold};
                ChCgPass<kCgPairB> f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.side[0] = x_cur;
                f.r_new = r_alt; f.p_new = pnew; f.x_new = x_alt; f.S = c->d_S;
                KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, PostCgOnePass{c->d_S, c->d_I, c->d_hist, c->hist_cap}));
                std::swap(r, r_alt);
                std::swap(x_cur, x_alt);
                std::swap(pold, pnew);
                z = r;
                continue;
            }
            if (onepass) {
                // pass 0 reads r_0 as p_0 as well; from then on p alternates between p1 (odd passes write it)
                // and p0
                ProfScope ps(c, 0, "cg_onepass (chain: r-=alpha*A p; p=r+beta*p; x+=alpha*p; A p; 4 dots)", 48.0 * n);
                Halo H{};
                const double *vecs[2] = {r, done + k == 0 ? r : pold};
                ChCg f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.side[0] = x_cur;
                f.r_new = r_alt; f.p_new = pnew; f.x_new = x_alt; f.S = c->d_S;
                KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, PostCgOnePass{c->d_S, c->d_I, c->d_hist, c->hist_cap}));
                std::swap(r, r_alt);
                std::swap(x_cur, x_alt);
                std::swap(pold, pnew);
                z = r;
                continue;
            }
            // ---- K1
            if (twice) {
                Halo H;
                const double *vecs[2] = {r, pold};
                const int it = done + k + 1, par_in = (it - 1) & 1, par_out = it & 1;
                if (push) {
                    for (int a = 0; a < 4; ++a) H.lo[a] = H.hi[a] = nullptr;
                    comm_push_recv(c, par_in, 0, &H.lo[0], &H.hi[0]);
                    comm_push_recv(c, par_in, 1, &H.lo[1], &H.hi[1]);
                } else {
                    KL_TRY(halo_exchange(&P, vecs, 2, &H));
                }
                {
                    ProfScope ps(c, 0, "cg_xdir_dot (stencil: x+=alpha_prev*p; p=r+beta*p; (A p).p)", 40.0 * n);
                    FCgDirX2 f;
                    set_io(f, &P, vecs, H);
                    set_gate(f, c, true);
                    f.p_new = pnew; f.x = x_cur; f.x_new = x_alt; f.S = c->d_S;
                    f.push_first = f.push_last = nullptr;
                    f.last_off = (size_t)(P.nyl - 1) * P.nx;
                    if (push) comm_push_send(c, par_out, 1, &f.push_first, &f.push_last);
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostCgAlpha{c->d_S}, true));
                    std::swap(x_cur, x_alt);
                }
#ifdef KL_TRACE
                if (getenv("KL_TRACE_K1") && it == maxit) continue;    // debug: leave K1's time stamps in g_trace
#endif
                {
                    ProfScope ps(c, 1, "cg_apply_rupdate_dot (stencil: r-=alpha*A(r+beta*p); r.r)", 24.0 * n);
                    FCgRUpdate f;
                    set_io(f, &P, vecs, H);      // same halo lines: r and p_old are unchanged since K1
                    set_gate(f, c, true);
                    f.r_new = r_alt; f.S = c->d_S;
                    f.push_first = f.push_last = nullptr;
                    f.last_off = (size_t)(P.nyl - 1) * P.nx;
                    if (push) comm_push_send(c, par_out, 0, &f.push_first, &f.push_last);
                    KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostCgEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap, 0}, true));
                }
                std::swap(r, r_alt);
                z = r;
                double *t = pold; pold = pnew; pnew = t;
                continue;
            }
            if (defer_x) {
                ProfScope ps(c, 0, "cg_xdir_apply_dot (stencil: x+=alpha_prev*p; p=z+beta*p; ax=A p; ax.p)", 48.0 * n);
                Halo H;
                const double *vecs[2] = {z, pold};
                KL_TRY(halo_exchange(&P, vecs, 2, &H));
                FCgDirX f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.p_new = pnew; f.ax = ax; f.x = dx; f.S = c->d_S;
                KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostCgAlpha{c->d_S}));
            } else if (fused) {
                ProfScope ps(c, 0, "cg_dir_apply_dot (stencil: p=z+beta*p; ax=A p; ax.p)", 32.0 * n);
                Halo H;
                const double *vecs[2] = {z, pold};
                KL_TRY(halo_exchange(&P, vecs, 2, &H));
                FCgDir f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.p_new = pnew; f.ax = ax; f.S = c->d_S;
                KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostCgAlpha{c->d_S}));
            } else {
                PAxpy u;
                set_gate(u, c, true);
                u.a = z; u.b = pold; u.y = pnew; u.S = c->d_S; u.s_idx = S_BETA; u.sign = 1.0;
                KL_TRY(launch_pointwise(c, u, n, NoPost{}));
                KL_TRY(op_apply(&P, pnew, ax, true));
                PDot2 d;
                set_gate(d, c, true);
                d.a = ax; d.b = pnew; d.c = nullptr; d.d = nullptr;
                KL_TRY(launch_pointwise(c, d, n, PostCgAlpha{c->d_S}));
            }
            // ---- K2 (+K3 fused for cbpr2)
            if (fuse_pc) {
                ProfScope ps(c, 3, "pcg_rupdate_precond (stencil: r-=alpha ax; z=cbpr2(r); r.r; r.z)", 32.0 * n);
                Halo H;
                const double *vecs[2] = {r, ax};
                KL_TRY(halo_exchange(&P, vecs, 2, &H));
                FPcgUpdateR f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true);
                f.r_new = r_alt; f.z = z; f.S = c->d_S; f.d = cf.d; f.calpha = cf.alpha;
                KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, PostCgEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap, 2}));
                std::swap(r, r_alt);
                double *t = pold; pold = pnew; pnew = t;
                continue;
            }
            if (defer_x) {
                ProfScope ps(c, 1, "cg_update_r_dot (pointwise: r-=alpha ax; r.r)", 24.0 * n);
                PCgUpdateR u;
                set_gate(u, c, true);
                u.r = r; u.ax = ax; u.S = c->d_S;
                KL_TRY(launch_pointwise(c, u, n, PostCgEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap, 0}));
                double *t = pold; pold = pnew; pnew = t;
                continue;
            }
            {
                ProfScope ps(c, 1, "cg_update_xr_dot (pointwise: x+=alpha p; r-=alpha ax; r.r)", 48.0 * n);
                PCgUpdate u;
                set_gate(u, c, true);
                u.x = dx; u.r = r; u.p = pnew; u.ax = ax; u.S = c->d_S;
                if (prec) KL_TRY(launch_pointwise(c, u, n, PostStoreRed{c->d_S, S_TMP0, 0}));
                else KL_TRY(launch_pointwise(c, u, n, PostCgEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap, 0}));
            }
            // ---- K3
            if (prec) {
                ProfScope ps(c, 2, "pcg_precond_dot (stencil: z=M^-1 r; r.z)", 16.0 * n);
                KL_TRY(pc_apply(&P, r, z, aux, aux2, 2, true,
                                PostCgEnd{c->d_S, c->d_I, c->d_hist, c->hist_cap, 1}));
            }
            double *t = pold; pold = pnew; pnew = t;
        }
        return KL_OK;
    };
    const bool use_graph = c->opt_use_graph && !c->opt_profile && c->nranks == 1 && fused &&
                           (P.pc.kind == KL_PC_NONE || P.pc.kind == KL_PC_CBPR2 || P.pc.kind == KL_PC_CHEB);
    while (done < maxit) {
        int batch = c->opt_check_every;
        if (batch > maxit - done) batch = maxit - done;
        Ctx::GraphEntry *ge = nullptr;
        // groups: the buffer roles alternate once per group, so a replayable batch (whose replay does not run the
        // host-side swaps of enqueue_iterations) is an even number of whole groups from phase 0 on.  Batches starting
        // mid-group run eagerly.
        const int period = group ? G : 2;
        if (use_graph && batch % (group ? 2 * G : 2) == 0 && done % period == 0) {
            GraphKey gk;
            gk.add('C').add(nx).add(ny).add(batch).add(P.op.kind).add(P.op.eps_x).add(P.op.eps_y).add(P.w5).add(P.pc.kind)
                .add(P.pc.degree).add(P.params).add(c->opt_tma).add(c->opt_chain).add(c->opt_stencil_rows)
                .add(c->opt_stencil_tail).add(c->opt_stencil_stagger).add(c->opt_pdl).add(c->opt_reverse).add(c->opt_persistent)
                .add(c->ws).add(dx).add(r).add(pold)
                .add(x_cur).add(cg_pass).add(onepass && done == 0)      // (one-pass: iteration 1 reads r as p)
                .add(group ? G : 0).add(done % period);
            ge = graph_find(c, gk.s);
            if (!ge && polls >= 1) {     // the first batch of a handle's first solve runs eagerly
                const long long l0 = c->stats.kernel_launches;
                KL_TRY(graph_begin(c));
                const int rc = enqueue_iterations(done, batch);
                if (rc < 0) {
                    Ctx::GraphEntry *dummy = nullptr;
                    graph_end(c, std::string(), 0.0, 0, &dummy);
                    graph_clear(c);
                    return rc;
                }
                KL_TRY(graph_end(c, gk.s, 0.0, c->stats.kernel_launches - l0, &ge));
                c->stats.kernel_launches = l0;
            }
        }
        if (ge) {
            KL_CUDA(c, cudaGraphLaunch(ge->exec, c->stream));
            c->stats.kernel_launches += ge->launches;
        } else {
            KL_TRY(enqueue_iterations(done, batch));
        }
        done += batch;
        KL_TRY(read_back(c));
        ++polls;
        if (c->h_pinned_i[I_CONV_AT] >= 0) {
            status = c->h_pinned_i[I_BREAKDOWN] ? KL_BREAKDOWN : KL_OK;
            break;
        }
    }
    if (group) {
        // after `its` passes (the passes after the convergence step were gated off), m = its / G groups stored x_{mG}
        // in x_start (m even) or the other buffer (m odd).  A group truncated by maxit stored x_{its} into dx.  If its
        // pass j < G raised the flag, one ungated store pass of depth j from the group's r_k, p_k, x_k forms x_{its}.
        if (status == KL_NOT_CONVERGED) KL_TRY(read_back(c));     // (maxit = 0: no poll ran)
        const int its_done = c->h_pinned_i[I_ITER], m = its_done / G, j = its_done % G;
        const double *xres = (m & 1) ? x_other : x_start;
        if (j != 0 && its_done == maxit) {
            xres = (m & 1) ? x_start : x_other;
        } else if (j != 0) {
            ProfScope ps(c, 7, kCgFinishName, 48.0 * n);
            double *xo = (m & 1) ? x_start : x_other;
            KL_TRY(cg_look(c, &P, j, true, (m & 1) ? r_other : r_start, (m & 1) ? p1 : p0, xres,
                           (m & 1) ? r_start : r_other, (m & 1) ? p0 : p1, xo, 1, false));
            xres = xo;
        }
        if (xres != dx) KL_CUDA(c, cudaMemcpyAsync(dx, xres, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    } else if (pair) {
        // after `its` passes (the passes after the convergence step were gated off) x_{2m}, m = its / 2, is in
        // x_start (m even) or the other buffer (m odd), and p_{2m} in p0 (m even) or p1 (m odd).  An odd `its` ended
        // on a pass A: x_{its} = x_{2m} + alpha_{2m} p_{2m}, the one-pass path's fma, with alpha_{2m} in
        // S_ALPHA_HIST.
        if (status == KL_NOT_CONVERGED) KL_TRY(read_back(c));     // (maxit = 0: no poll ran)
        const int its_done = c->h_pinned_i[I_ITER], m = its_done / 2;
        const double *xres = (m & 1) ? x_other : x_start;
        if (its_done & 1) {
            PAxpy u;
            set_gate(u, c, false);
            u.a = xres; u.b = (m & 1) ? p1 : p0; u.y = dx; u.S = c->d_S; u.s_idx = S_ALPHA_HIST; u.sign = 1.0;
            KL_TRY(launch_pointwise(c, u, n, NoPost{}));
        } else if (xres != dx) {
            KL_CUDA(c, cudaMemcpyAsync(dx, xres, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        }
    } else if (onepass) {
        // no deferred update: after `its` passes x is in x_start (even) or the other buffer (odd); the passes
        // after the convergence step were gated off
        if (status == KL_NOT_CONVERGED) KL_TRY(read_back(c));     // (maxit = 0: no poll ran)
        const int its_done = c->h_pinned_i[I_ITER];
        const double *xres = (its_done & 1) ? x_other : x_start;
        if (xres != dx) KL_CUDA(c, cudaMemcpyAsync(dx, xres, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    } else if (defer_x) {
        // flush the pending x += alpha p of the last executed iteration (kernels after the convergence step
        // were gated off, so S_ALPHA and the p buffer of that iteration are intact).  Iteration i wrote its
        // direction into p1 for odd i and into p0 for even i.
        if (status == KL_NOT_CONVERGED) KL_TRY(read_back(c));
        const int its_done = c->h_pinned_i[I_ITER];
        if (its_done > 0) {
            // `twice`: x is ping-ponged; K1 of iteration i read buffer (i-1)&1 and wrote buffer i&1 (0 = dx), and
            // the K1 launches after the convergence step did nothing: the current x is in buffer its_done&1.
            const double *xsrc = (twice && (its_done & 1)) ? ((x_cur == dx) ? x_alt : x_cur) : dx;
            PAxpy u;
            set_gate(u, c, false);
            u.a = xsrc; u.b = (its_done & 1) ? p1 : p0; u.y = dx; u.S = c->d_S; u.s_idx = S_ALPHA; u.sign = 1.0;
            KL_TRY(launch_pointwise(c, u, n, NoPost{}));
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
    // groups: 16n B per pass that stores nothing, 48n B per store pass; a group cut short by maxit ends on a store
    // pass, one cut short by convergence on a pass that stores nothing and the finishing store pass
    const int gt = group ? its % G : 0;
    c->stats.algorithmic_bytes =
        group ? (double)(its / G) * (16.0 * (G - 1) + 48.0) * (double)n +
                    (gt == 0 ? 0.0 : (16.0 * (its == maxit ? gt - 1 : gt) + 48.0) * (double)n)
        : pair ? (24.0 * ((its + 1) / 2) + 48.0 * (its / 2) + 24.0 * (its & 1)) * (double)n
                                      : (double)its * (fuse_pc ? 80.0 : (prec ? 96.0 : (onepass ? 48.0 : (twice ? 64.0 : (defer_x ? 72.0 : 80.0))))) * (double)n;
    *res_out = c->h_pinned[S_RES];
    if (status == KL_OK) *iter = c->h_pinned_i[I_CONV_AT];   // count on exit; unchanged if not converged
    return status;
}

}  // namespace kl

using namespace kl;

extern "C" {

#ifdef KL_TRACE
// debug: time stamps of the CTAs of the last stencil kernel launched from this file (3 u64 per CTA + 1)
int kl_debug_trace_cg(unsigned long long *out, int n) {
    return cudaMemcpyFromSymbol(out, g_trace, sizeof(unsigned long long) * n) == cudaSuccess ? 0 : -1;
}
#endif

int kl_cg(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny, double tol,
          int *iter, double *res) {
    return cg_solve(h, A, b, x, nx, ny, tol, iter, res, nullptr, nullptr, 0);
}
int kl_cg_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
              double tol, int *iter, double *res) {
    return cg_solve(h, A, b, x, nx, ny, tol, iter, res, nullptr, nullptr, 0);
}
int kl_pcg(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny, double tol,
           int *iter, double *res, const kl_precond_t *M, const double *params, int nparams) {
    return cg_solve(h, A, b, x, nx, ny, tol, iter, res, M, params, nparams);
}
int kl_pcg_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
               double tol, int *iter, double *res, const kl_precond_t *M, const double *params,
               int nparams) {
    return cg_solve(h, A, b, x, nx, ny, tol, iter, res, M, params, nparams);
}

}  // extern "C"
