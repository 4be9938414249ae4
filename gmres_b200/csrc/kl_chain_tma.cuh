// kl_chain_tma.cuh -- temporally blocked ("chained") marching stencil kernel (sm_100a).
//
// L dependent applications of the 5-point operator in ONE pass over HBM: the
// degree-k Chebyshev preconditioner (k applications; ChCheb / ChChebCont below)
// and BiCGSTAB's "update -> cbpr2 -> operator -> dot products" steps (ChBiDir,
// ChBiS in kl_bicgstab.cu) read their inputs once and write their outputs once,
// no matter how many operator applications lie in between.  Measured (8192^2,
// DESIGN.md section 6): DRAM traffic = inputs + outputs (ncu), degree 4 in 441 us
// against 1601 us for four passes; the kernel is issue-bound, not HBM-bound,
// beyond L = 1 (~50 instructions per level and warp-line, 16 of them FP64).
//
// Geometry.  A CTA of 4 warps owns a strip of 4*(64-2H) columns, H = L rounded
// up to even, and marches down `rows` grid lines.  Every WARP is independent: it
// owns a 64-column window (lane l: window columns 2l, 2l+1) whose outer H
// columns are halo -- level l of the chain is valid on window columns
// [l, 64-l), so left/right neighbours always come from warp shuffles and no
// inter-warp exchange or CTA barrier is needed inside the march.  In the march
// direction level l runs l lines behind level 0: when input line R arrives,
// level l produces line R-l from lines R-l-1, R-l, R-l+1 of level l-1, which sit
// in registers (3-line window per level, rotated by compile-time phase: the
// march is unrolled 6 = lcm(3,2) lines so no register moves are executed).  A
// CTA therefore reads rows+2L lines to write rows lines; overlapping lines and
// columns are L2 hits (neighbouring CTAs run concurrently), DRAM sees every
// input once.
//
// Input lines arrive through a ring of shared-memory stages filled by 2-D TMA
// box loads (box = BWP columns x SR lines per input array, full/empty mbarrier
// pair per stage, one elected producer thread).  The ring keeps the last L lines
// alive, so level l re-reads raw inputs (e.g. the Chebyshev right-hand side r)
// at its own line with one LDS.128 instead of carrying them through registers.
// TMA's out-of-bounds zero fill supplies the zero-Dirichlet boundary for level
// 0; levels >= 1 are forced to zero outside the domain (those points are not
// unknowns).
//
// Multi-GPU (template parameter MG): the L lines above / below the slab come from
// the neighbours' halo buffers (kl_ops.cu halo_exchange_lines) and are patched
// into the ring by the thread that reads them; the neighbours' lines are
// recomputed redundantly level by level, so one exchange serves the whole chain.
//
// Chain functor contract (see ChCheb below and ChBiDir / ChBiS in kl_bicgstab.cu):
//   NIN, L, NC, NRED               inputs, levels, carried values per point, reductions
//   void init()
//   void level0(bool out, size_t idx, const double (&raw)[NIN][2], double (&u)[2], double (&cc)[NC][2], double *acc)
//        u = level-0 field at the two points of this thread, cc = carried values;
//        `out`: the points are in the CTA's output range (store level-0 outputs)
//   template <class RAW>
//   void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
//              const double (&cin)[NC][2], RAW raw, const double (&sd)[max(NSIDE,1)][2], double (&u)[2],
//              double (&cout)[NC][2], double *acc)
//        lv in 1..L ; up = field of level lv-1, au = A up ; raw(a) = double2 of input a at this line ;
//        sd = side inputs (arrays side[0..NSIDE), read point-wise at the last level's output points only,
//        valid for lv == L && out; the kernel prefetches them two lines ahead into registers)
// level0 must map all-zero inputs to u = 0 (outside the domain TMA delivers zeros).
// VAROP functors (ChJacCheb) take the diagonal of A at their points as well: level0(out, idx, raw, dg, u, cc, acc)
// and level(lv, out, idx, up, au, dg, cin, raw, sd, u, cout, acc); their level-0 values outside the domain never
// reach the domain (the checked march applies the boundary rule to neighbours).
#pragma once
#include <type_traits>

#include "kl_stencil_tma.cuh"

namespace kl {

constexpr int kChainWarps = 4;
constexpr int kChainThreads = kChainWarps * 32;
constexpr int kChainMaxL = 6;

// VAR: the variable-coefficient operator needs one more halo column (its level 0 reads kx at columns -1 and +1)
template <int L, bool VAR = false>
struct ChainDims {
    static constexpr int H = (L + (VAR ? 1 : 0) + 1) & ~1;   // halo columns per window side
    static constexpr int WW = 64 - 2 * H;               // output columns per warp
    static constexpr int STRIP = kChainWarps * WW;      // output columns per CTA
    static constexpr int BW = STRIP + 2 * H;            // columns a CTA needs
    static constexpr int BWP = (BW + 15) & ~15;         // TMA box width (row pitch multiple of 128 B)
};
// Ring geometry: SR lines per stage, NST stages (defaults in ChainBase, a functor may override them).  The
// ring holds NR = SR*NST lines (a multiple of 6: the march is unrolled by hexads) and keeps RET stages alive
// behind the current one so that level l can re-read raw inputs l lines back.
template <class C>
struct ChainRing {
    static constexpr int SR = C::SR;
    static constexpr int NST = C::NST;
    static constexpr int NR = SR * NST;
    static constexpr int RET = (C::LAG * C::L + (C::VAROP ? 2 : 0) + SR - 1) / SR;
    static constexpr int P = 6;                         // unroll period of the march = lcm(3 field slots, 2 carried slots)
    static_assert(P % SR == 0, "an unroll period must hold whole stages");
    static_assert(NR % P == 0, "ring must hold whole periods");
    static_assert(NST - RET >= 2, "ring too shallow");
    static constexpr size_t bytes = (size_t)C::NIN * NR * ChainDims<C::L, C::VAROP>::BWP * sizeof(double) + 2 * NST * 8 + 64;
};

struct ChainGeo {
    int nx, ny, rows;
    int row_lo, row_hi;    // lines of the domain this rank can see: [row_lo, row_hi) (single GPU: 0, ny)
};

template <int NIN_, int L_, int NC_, int NRED_>
struct ChainBase {
    static constexpr int NIN = NIN_;
    static constexpr int L = L_;
    static constexpr int NC = NC_;
    static constexpr int NRED = NRED_;
    static constexpr int NSIDE = 0;     // point-wise side inputs of the last level, prefetched 2 lines ahead
    // VAROP: the chain applies KL_OP_ANISO5_VAR with in[1] = kx, in[2] = ky (see "Variable coefficients" above
    // k_chain_tma); the functor's level0 / level then also receive the diagonal of A
    static constexpr bool VAROP = false;
    // SINGLE_GPU: no multi-GPU instantiation (a functor whose solver path runs on one GPU only)
    static constexpr bool SINGLE_GPU = false;
    // LAG: how many lines level l runs behind level l-1.  With LAG = 1 level l consumes the line level l-1
    // produced in the SAME march step, so a step is one dependent chain of 7L FP64 operations (~250 cycles of
    // latency at L = 4 with 4 warps per scheduler to hide it: the round-1 kernel ran the FP64 pipe at 44 %).
    // With LAG = 2 every level reads only lines finished in EARLIER steps: the L levels of a step are
    // independent instruction streams (processed last level first, so a level reads its predecessor's window
    // before the predecessor overwrites the oldest line -- still 3 lines per level).  Price: L more march steps
    // per CTA and 2L instead of L lines of ring retention, which is why multi-input chains keep LAG = 1.
    // Measured at 8192^2 (profiles/r02_bench_chain_cheb8192.txt): LAG 2 wins only at L = 2 (232 vs 245 us); from
    // L = 4 on its extra address arithmetic and spills under the register cap cost more than the latency it hides
    // (L = 5: 667 vs 524 us).
#ifdef KL_CHAIN_LAG
    static constexpr int LAG = NIN_ == 1 ? KL_CHAIN_LAG : 1;
#else
    static constexpr int LAG = (NIN_ == 1 && L_ == 2) ? 2 : 1;
#endif
    // LEAN: interior CTAs run their middle hexads through a copy of the march without out-of-domain masks (see
    // k_chain_tma).  Pays from L = 3 on (L - 1 masked levels; 322 -> 292 us at L = 3, 703 -> 643 us at L = 6); at
    // L <= 2 the checked first hexad it needs costs more than the masks (+9 %; BiCGSTAB's two-level chains included).
    // The three-input continuation chunks (L >= 3) gain like the single-input ones: degree 8 = 4 + 4: ~1040 -> 940 us.
    static constexpr bool LEAN = L_ >= 3;     // (also the three-input continuation chunks of degrees 7..12)
    // Two columns per thread.  A four-column variant (half the shuffles and per-line overhead per point, but
    // ~160 registers at L = 2, i.e. 3 CTAs per SM instead of 6) measured 10-50 % slower: these kernels are
    // dependent FP64 chains behind a shuffle and live on thread-level parallelism.
    // ring: 1 input: 3-line stages, 18 / 24 lines ; more inputs: 1-line stages, 6 lines (a CTA needs ~2 us per
    // line, so three lines of lookahead cover the DRAM latency; small rings buy 6 CTAs per SM instead)
    static constexpr int SR = NIN_ == 1 ? 3 : 1;
    static constexpr int NST = NIN_ == 1 ? (L_ <= 2 ? 6 : 8) : 6;
    static constexpr int MINB = L_ <= 2 ? 6 : (L_ <= 4 ? 4 : 3);   // CTAs per SM the register budget is cut for
    static_assert(L_ >= 1 && L_ <= kChainMaxL, "chain length");
    const double *in[NIN_];
    const double *lo[NIN_];     // multi-GPU: the neighbours' L boundary lines of every input (nullptr at the
    const double *hi[NIN_];     // global boundary): lo = grid lines -L..-1, hi = lines ny..ny+L-1
    const double *side[1];
    const int *flags;
    int step;
    int run_on_conv;
    OpCoef coef;
    __device__ __forceinline__ bool skip() const {
        if (!flags) return false;
        int ca = flags[I_CONV_AT];
        return !(ca < 0 || (run_on_conv && ca == step));
    }
};

__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 5-point operator, same rounding as apply5 with one instruction less: 4*c is exact, so
// fma(4, c, -s) == 4*c - s bit for bit (poisson.f90:42, :88-92).
template <int OPK>
__device__ __forceinline__ double apply5c(double c, double l, double r, double dn, double up, const OpCoef &k) {
    if (OPK == KL_OP_POISSON5) {
        return fma(4.0, c, -(((l + r) + dn) + up));
    } else if (OPK == KL_OP_POISSON5_BRANCHY) {
        return ((fma(4.0, c, -l) - r) - up) - dn;
    } else if (OPK == KL_OP_STENCIL5) {
        double s = fma(k.ex, l, k.exr * r), t = fma(k.ey, dn, k.eyu * up);
        return fma(k.cc, c, -(s + t));
    } else {
        double sx = l + r, sy = dn + up;
        double t = fma(k.ex, sx, k.ey * sy);
        return fma(k.cc, c, -t);
    }
}

// Variable coefficients (C::VAROP, OPK = KL_OP_ANISO5_VAR, one GPU): every level computes its face weights from the
// ring -- kx of its own line (columns -1 and +2 by shuffle), ky of lines rho-1, rho, rho+1 -- and hands A u and the
// diagonal to the functor; level 0 gets the diagonal of its line too (for D^-1 r).  So that level 0 can see ky one
// line ahead, ky is loaded one line down (ring line R holds ky line R+1; TMA zero-fills line ny), the march starts
// two lines earlier (the ring's first ky line is then two lines above the first level-0 line that counts) and the
// ring keeps two more lines.  Level 0 also needs kx one column outside its window, hence one more halo column
// (ChainDims<L, true>).  The zeros TMA delivers outside the domain are not the boundary rule (a boundary face takes
// the cell's own coefficient): the checked copy of the march applies the rule, lean hexads lie strictly inside the
// domain and need none.
// Face weights, diagonal and (AU) au = A u at the thread's two points of line `row`, same evaluation order as
// oracle/krylov_extras.c ko_aniso_var.  u: cu = line row, up = row-1, dn = row+1.  All lanes must call it.
template <bool AU, bool CHK>
__device__ __forceinline__ void var_apply(const double2 kx, const double2 kyu, const double2 kyc, const double2 kyd,
                                          const double (&cu)[2], const double (&up)[2], const double (&dn)[2],
                                          const int gc, const int row, const int nx, const int ny, double (&au)[2],
                                          double (&dg)[2]) {
    const double kxs[4] = {__shfl_up_sync(0xffffffffu, kx.y, 1), kx.x, kx.y, __shfl_down_sync(0xffffffffu, kx.x, 1)};
    double xs[4] = {0.0, cu[0], cu[1], 0.0};
    if (AU) {
        xs[0] = __shfl_up_sync(0xffffffffu, cu[1], 1);
        xs[3] = __shfl_down_sync(0xffffffffu, cu[0], 1);
    }
    const double ku[2] = {kyu.x, kyu.y}, kc[2] = {kyc.x, kyc.y}, kd[2] = {kyd.x, kyd.y};
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int i = gc + e;
        const bool hl = !CHK || i > 0, hr = !CHK || i < nx - 1, hu = !CHK || row > 0, hd = !CHK || row < ny - 1;
        const double kxc = kxs[e + 1];
        const double wl = hl ? 0.5 * (kxc + kxs[e]) : kxc, wr = hr ? 0.5 * (kxc + kxs[e + 2]) : kxc;
        const double wu = hu ? 0.5 * (kc[e] + ku[e]) : kc[e], wd = hd ? 0.5 * (kc[e] + kd[e]) : kc[e];
        dg[e] = ((wl + wr) + wd) + wu;
        if (AU) {
            const double xl = hl ? xs[e] : 0.0, xr = hr ? xs[e + 2] : 0.0;
            const double xu = hu ? up[e] : 0.0, xd = hd ? dn[e] : 0.0;
            const double s = fma(wl, xl, wr * xr), t = fma(wd, xd, wu * xu);
            au[e] = fma(dg[e], cu[e], -(s + t));
        }
    }
}

// MG: multi-GPU instantiation (lines above / below the slab come from the neighbours' halo buffers).  It is a
// template parameter because the patch code in the level-0 path (global loads + ring stores in all six unrolled
// phases) cost the single-GPU kernels 10-28 % when it was a run-time branch.
template <class C, int OPK, bool MG>
__global__ void __launch_bounds__(kChainThreads, C::MINB)
k_chain_tma(const C c_in, const ChainGeo g, const RedCtl rc, const __grid_constant__ TMaps<C::NIN> tm) {
    if (c_in.skip()) return;
    C f = c_in;
    f.init();
    constexpr int NIN = C::NIN, L = C::L, NC = C::NC, NRED = C::NRED;
    constexpr int NR_ = NRED > 0 ? NRED : 1;
    static_assert(C::VAROP == (OPK == KL_OP_ANISO5_VAR) && (!C::VAROP || (NIN == 3 && !MG)), "variable-coefficient chain");
    // variable coefficients: the march starts VX lines earlier -- ky is loaded one line down, so the first ky line
    // in the ring is jstart + 1, and level 0 at line R needs ky line R - 1: level 0 is valid from jstart + 2 on
    constexpr int VX = C::VAROP ? 2 : 0;
    using D = ChainDims<L, C::VAROP>;
    using RG = ChainRing<C>;
    constexpr int NSIDE = C::NSIDE, NSD = NSIDE > 0 ? NSIDE : 1;
    constexpr int H = D::H, WW = D::WW, BWP = D::BWP;
    constexpr int SR = RG::SR, NST = RG::NST, NR = RG::NR, RET = RG::RET, LAG = C::LAG;
    static_assert(LAG == 1 || LAG == 2, "level lag");
    // Unroll period P and carried-value slots CCS.  The carried values of a point (e.g. the Chebyshev direction d)
    // are consumed LAG steps after they were produced: with LAG 1 the consumer runs after the producer within a
    // step (old and new value live at once), with LAG 2 the value must survive two steps -- two slots either way,
    // rotation period lcm(3, 2) = 6.  (A period-3 march needs a third carried slot, 4 L NC more registers, which the
    // 128-register budget at L = 3, 4 does not have.)
    constexpr int P = RG::P, CCS = 2;
    constexpr int NB = (LAG * L + (C::VAROP ? 2 : 0) + P - 1) / P;   // how many periods back raw inputs are re-read
    constexpr unsigned kStageBytes = NIN * SR * BWP * sizeof(double);

    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *ring = reinterpret_cast<double *>(smem_raw);                       // [NIN][NR][BWP]
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem_raw + (size_t)NIN * NR * BWP * sizeof(double));
    unsigned long long *empty = full + NST;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int i0 = blockIdx.x * D::STRIP;            // first output column of the CTA
    const int bc = wid * WW + 2 * lane;              // this thread's column pair inside the box
    const int gc = i0 - H + bc;                      // ... and in the grid
    const bool colin0 = gc >= 0 && gc < g.nx, colin1 = gc + 1 >= 0 && gc + 1 < g.nx;
    const bool outlane = lane >= H / 2 && lane < 32 - H / 2 && gc < g.nx;
    const int j0 = blockIdx.y * g.rows;
    const int j1 = min(j0 + g.rows, g.ny);
    const int jstart = j0 - L - VX;                  // grid line of march step 0
    const int T = (j1 - j0) + L + LAG * L + VX;      // march steps (level L emits line R - LAG*L)
    const int nstg = (T + SR - 1) / SR;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NST; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kChainWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int q) {
        const int s = q % NST;
        mbar_expect_tx(&full[s], kStageBytes);
#pragma unroll
        for (int a = 0; a < NIN; ++a)
            tma_load_2d(ring + ((size_t)a * NR + (size_t)s * SR) * BWP, &tm.m[a], &full[s], i0 - H,
                        jstart + q * SR + ((C::VAROP && a == 2) ? 1 : 0));
    };
    if (tid == 0) {
        for (int q = 0; q < NST && q < nstg; ++q) issue(q);
    }

    double acc[NR_];
#pragma unroll
    for (int k = 0; k < NR_; ++k) acc[k] = 0.0;
    // register windows: U[l][slot][e] = field of level l (l < L), 3 lines ; CC[l][slot][k][e] carried values, 2 lines
    double U[L][3][2], CC[L][CCS][NC][2];
#pragma unroll
    for (int l = 0; l < L; ++l) {
#pragma unroll
        for (int s = 0; s < 3; ++s) U[l][s][0] = U[l][s][1] = 0.0;
#pragma unroll
        for (int s = 0; s < CCS; ++s)
#pragma unroll
            for (int k = 0; k < NC; ++k) CC[l][s][k][0] = CC[l][s][k][1] = 0.0;
    }

    double SD[NSD][3][2];             // side inputs of the last level: lines rho, rho+1, rho+2
#pragma unroll
    for (int a = 0; a < NSD; ++a)
#pragma unroll
        for (int s = 0; s < 3; ++s) SD[a][s][0] = SD[a][s][1] = 0.0;

    const double *tb = ring + bc;     // this thread's pair in ring line 0 of input 0
    const double *rbase[NB + 1];      // ring line of the current period [0] and of the NB periods before it
#pragma unroll
    for (int k = 0; k <= NB; ++k) rbase[k] = tb;
    const double *&cur = rbase[0];
    int q = 0;                        // stage of the current march step
    // input a at ring line (current period + kk), kk >= -NB*P (compile time after unrolling)
    auto ring_at = [&](int a, int kk) -> double2 {
        const int bk = kk >= 0 ? 0 : (-kk + P - 1) / P;
        return *reinterpret_cast<const double2 *>(rbase[bk] + ((size_t)a * NR + (size_t)(kk + bk * P)) * BWP);
    };

    // one march step; PH = step index mod 6 (compile time), t = step index.  LEAN: the step belongs to a hexad
    // in which the last level's line is inside [j0, j1) for all six steps, of a CTA whose windows and lines all
    // lie inside the domain (see `lean_cta` below): no out-of-domain masks, no halo-line patch, the output
    // predicate of the last level is the loop-invariant `outlane` (12 FSEL and ~12 ISETP/PLOP3 less per step at
    // L = 4).  Everything else -- first and last hexads, CTAs on the domain edge -- takes the generic path.
    auto step = [&](auto ph, auto lean_c, const int t) {
        constexpr int PH = decltype(ph)::value;
        constexpr bool LEAN = decltype(lean_c)::value;
        const int R = jstart + t;     // grid line entering level 0
        if (NSIDE > 0) {
            // the last level reaches line R - L + 2 two steps from now: start its point-wise loads today
            const int rho2 = R - LAG * L + 2;
            if (outlane && rho2 >= j0 && rho2 < j1) {
#pragma unroll
                for (int a = 0; a < NSIDE; ++a) {
                    const double2 v = ldg2(f.side[a] + (size_t)rho2 * g.nx + gc);
                    SD[a][(PH + 2) % 3][0] = v.x;
                    SD[a][(PH + 2) % 3][1] = v.y;
                }
            }
        }
        // ---- level 0 -------------------------------------------------------
        auto level_zero = [&]() {
            double raw[NIN][2];
            if (MG && !LEAN && ((R < 0 && f.lo[0] != nullptr) || (R >= g.ny && R < g.ny + L && f.hi[0] != nullptr))) {
                // multi-GPU: this line belongs to a neighbour rank; TMA delivered zeros, take it from the halo
                // buffer and patch the ring (every thread re-reads only its own column pair later)
#pragma unroll
                for (int a = 0; a < NIN; ++a) {
                    const double *src = R < 0 ? f.lo[a] + (size_t)(R + L) * g.nx : f.hi[a] + (size_t)(R - g.ny) * g.nx;
                    raw[a][0] = colin0 ? __ldg(src + gc) : 0.0;
                    raw[a][1] = colin1 ? __ldg(src + gc + 1) : 0.0;
                    *reinterpret_cast<double2 *>(const_cast<double *>(cur) + ((size_t)a * NR + PH) * BWP) =
                        make_double2(raw[a][0], raw[a][1]);
                }
            } else {
#pragma unroll
                for (int a = 0; a < NIN; ++a) {
                    const double2 v = *reinterpret_cast<const double2 *>(cur + ((size_t)a * NR + PH) * BWP);
                    raw[a][0] = v.x;
                    raw[a][1] = v.y;
                }
            }
            const bool out = outlane && R >= j0 && R < j1;
            if constexpr (C::VAROP) {
                double dg[2], au_unused[2];
                var_apply<false, !LEAN>(ring_at(1, PH), ring_at(2, PH - 2), ring_at(2, PH - 1), ring_at(2, PH),
                                        U[0][PH % 3], U[0][PH % 3], U[0][PH % 3], gc, R, g.nx, g.ny, au_unused, dg);
                f.level0(out, (size_t)R * g.nx + gc, raw, dg, U[0][PH % 3], CC[0][PH % CCS], acc);
            } else {
                f.level0(out, (size_t)R * g.nx + gc, raw, U[0][PH % 3], CC[0][PH % CCS], acc);
            }
        };
        if (LAG == 1) level_zero();
        // ---- levels 1..L (LAG 1: ascending, each consumes what its predecessor just produced; LAG 2: descending,
        //      all independent, each reads its predecessor's window before the predecessor rotates it) -------------
#pragma unroll
        for (int li = 0; li < L; ++li) {
            const int l = LAG == 1 ? li + 1 : L - li;
            const int sl_cu = (PH - LAG * l + 24) % 3;          // slot of line rho = R - LAG*l in U[l-1]
            const int sl_up = (PH - LAG * l - 1 + 24) % 3;      // line rho-1
            const int sl_dn = (PH - LAG * l + 1 + 24) % 3;      // line rho+1
            const int cs_in = (PH - LAG * l + 24) % CCS;        // slot of line rho in CC[l-1]
            const int rho = R - LAG * l;
            const double(&cu)[2] = U[l - 1][sl_cu];
            const double(&up)[2] = U[l - 1][sl_up];
            const double(&dn)[2] = U[l - 1][sl_dn];
            double au[2], dg[2];
            // raw inputs of line rho from the ring (an earlier hexad when PH < LAG*l)
            const int kb = PH - LAG * l;
            if constexpr (C::VAROP) {
                // ring line m of ky holds ky line m+1
                var_apply<true, !LEAN>(ring_at(1, kb), ring_at(2, kb - 2), ring_at(2, kb - 1), ring_at(2, kb), cu, up, dn,
                                       gc, rho, g.nx, g.ny, au, dg);
            } else {
                double lf = __shfl_up_sync(0xffffffffu, cu[1], 1);
                double rt = __shfl_down_sync(0xffffffffu, cu[0], 1);
                au[0] = apply5c<OPK>(cu[0], lf, cu[1], dn[0], up[0], f.coef);
                au[1] = apply5c<OPK>(cu[1], cu[0], rt, dn[1], up[1], f.coef);
            }
            const int back = kb >= 0 ? 0 : (-kb + P - 1) / P;    // periods back (compile time after unrolling)
            const double *rb = rbase[back] + (size_t)(kb + back * P) * BWP;
            auto rawget = [&](int a) -> double2 {
                return *reinterpret_cast<const double2 *>(rb + (size_t)a * NR * BWP);
            };
            const bool out = (LEAN && l == L) ? outlane : (outlane && rho >= j0 && rho < j1);
            double un[2], cn[NC][2];
            double sd[NSD][2];
#pragma unroll
            for (int a = 0; a < NSD; ++a) {
                sd[a][0] = SD[a][PH % 3][0];
                sd[a][1] = SD[a][PH % 3][1];
            }
            if constexpr (C::VAROP) f.level(l, out, (size_t)rho * g.nx + gc, cu, au, dg, CC[l - 1][cs_in], rawget, sd, un, cn, acc);
            else f.level(l, out, (size_t)rho * g.nx + gc, cu, au, CC[l - 1][cs_in], rawget, sd, un, cn, acc);
            if (l < L) {
                const bool rowin = LEAN || (rho >= g.row_lo && rho < g.row_hi);
                const bool m0 = LEAN || (rowin & colin0), m1 = LEAN || (rowin & colin1);
                const int sl_new = (PH - LAG * l + 24) % 3;     // line rho in U[l]
                const int cs_new = (PH - LAG * l + 24) % CCS;
                U[l < L ? l : 0][sl_new][0] = m0 ? un[0] : 0.0;
                U[l < L ? l : 0][sl_new][1] = m1 ? un[1] : 0.0;
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    CC[l < L ? l : 0][cs_new][k][0] = cn[k][0];
                    CC[l < L ? l : 0][cs_new][k][1] = cn[k][1];
                }
            }
        }
        if (LAG != 1) level_zero();
    };

    // one stage boundary check + step, phase PH.  CHECK = false: the step is known to exist (whole hexads of the
    // main loop) -- no per-step bound test, so the march body is straight-line code and the shuffles need no
    // reconvergence scaffolding (WARPSYNC / ENDCOLLECTIVE around every SHFL of a conditionally executed step)
    auto phase = [&](auto ph, auto chk, auto lean_c, const int t) {
        constexpr int PH = decltype(ph)::value;
        constexpr bool CHECK = decltype(chk)::value;
        if (!CHECK || t < T) {
            if (PH % SR == 0) mbar_wait(&full[q % NST], (unsigned)((q / NST) & 1));
            step(ph, lean_c, t);
            if (PH % SR == SR - 1) {
                // this warp is done with stage q - RET (its lines are more than L behind the next step)
                __syncwarp();
                if (q >= RET) {
                    const int qs = q - RET;
                    if (lane == 0) mbar_arrive(&empty[qs % NST]);
                    if (tid == 0 && qs + NST < nstg) {
                        mbar_wait(&empty[qs % NST], (unsigned)((qs / NST) & 1));
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        issue(qs + NST);
                    }
                }
                ++q;
            }
        }
    };
    using TT = std::true_type;
    using FF = std::false_type;

    // a CTA is lean when every column of its four windows and every line it touches is inside the domain
    // (variable coefficients: and VX lines below, so that no line a lean hexad reads ky from is a boundary line)
    const bool lean_cta = i0 - H >= 0 && i0 - H + kChainWarps * WW + 2 * H <= g.nx && jstart >= 0 && jstart + T + VX <= g.ny;
    constexpr int kLeanT0 = L + LAG * L + VX; // first step whose last-level line is >= j0

    // Two copies of the march per kernel: a fast one for whole hexads and the generic, step-by-step checked one.
    //   LEAN kernels : fast = lean hexads of interior CTAs ; generic = first hexads, the partial last one, edge CTAs
    //   others       : fast = every whole hexad (generic but unchecked) ; checked = the partial last hexad
    using LeanT = std::integral_constant<bool, C::LEAN>;
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;
    using I3 = std::integral_constant<int, 3>;
    using I4 = std::integral_constant<int, 4>;
    using I5 = std::integral_constant<int, 5>;
    int hs = 0;   // ring line of the current period
    auto set_period = [&]() {
#pragma unroll
        for (int k = 0; k <= NB; ++k) {
            int h = hs - k * P;
            if (h < 0) h += NR;
            rbase[k] = tb + (size_t)h * BWP;
        }
    };
    // P phases with the given CHECK / LEAN flags
    auto period = [&](auto chk, auto lean_c, const int t0) {
        phase(I0{}, chk, lean_c, t0 + 0);
        phase(I1{}, chk, lean_c, t0 + 1);
        phase(I2{}, chk, lean_c, t0 + 2);
        if (P == 6) {
            phase(I3{}, chk, lean_c, t0 + 3);
            phase(I4{}, chk, lean_c, t0 + 4);
            phase(I5{}, chk, lean_c, t0 + 5);
        }
    };
    if (C::LEAN) {
        for (int t0 = 0; t0 < T; t0 += P) {
            set_period();
#ifdef KL_CHAIN_LEAN_ONLY      /* instruction counting only (scripts/sass_loops.py): drops the generic copy */
            if (true) {
#else
            if (lean_cta && t0 >= kLeanT0 && t0 + P <= T) {
#endif
                period(FF{}, LeanT{}, t0);
            } else {
                period(TT{}, FF{}, t0);
            }
            hs += P;
            if (hs == NR) hs = 0;
        }
    } else {
        int t0 = 0;
        for (; t0 + P <= T; t0 += P) {
            set_period();
            period(FF{}, FF{}, t0);
            hs += P;
            if (hs == NR) hs = 0;
        }
        if (t0 < T) {
            set_period();
            period(TT{}, FF{}, t0);
        }
    }

    if (NRED > 0) {
        __shared__ double sm[NR_ * (kChainThreads / 32)];
        __shared__ int s_flag;
        block_sum<NR_, kChainThreads>(acc, sm);
        const unsigned nb = gridDim.x * gridDim.y, bid = blockIdx.y * gridDim.x + blockIdx.x;
        grid_sum<NR_, kChainThreads>(acc, rc, nb, bid, &s_flag, sm);
    }
}

// host: tensor map with an explicit box (kl_core.cu)
int tmap_encode_box(Ctx *c, CUtensorMap *out, const double *base, int nx, int ny, int box_x, int box_y);

// lines per CTA: the redundant work is 2L / rows; keep it below ~10 % but leave >= ~3 CTAs per SM.
template <int L, bool VAR = false>
inline bool chain_geometry(Ctx *c, int nx, int ny, ChainGeo *g, dim3 *grid, bool single_input = false) {
    const long gx = (nx + ChainDims<L, VAR>::STRIP - 1) / ChainDims<L, VAR>::STRIP;
    if (gx > kMaxBlocks) return false;
    // measured at 8192^2 (profiles/r02_chain_rows_sweep.txt): L <= 3 is flat between 24L and 64L lines; from L = 4 on
    // the single-input chains like longer marches (fewer redundant lines, more lean hexads): L = 4: 392 / 384 / 381 /
    // 398 / 429 us at 96 / 160 / 192 / 224 / 256 lines, L = 6: 683 / 628 / 596 / 630 / 648 us.  The multi-input chains
    // (continuation chunks, BiCGSTAB) run 2-3 CTAs per SM and lose more to the ragged last wave than they gain.
    long rows = c->opt_stencil_rows > 0 ? c->opt_stencil_rows : ((L <= 3 || !single_input) ? 24 * L : 192);
    if (rows < 24) rows = 24;
    const long want = (long)kNumSM * 4;
    // small grids are launch-/latency-bound: many short marches (redundant lines are free there) beat few long ones
    const long rmin = c->opt_chain_rows_min > 0 ? c->opt_chain_rows_min
                                                : ((long)nx * ny <= (1L << 18) ? 6 : (12 * L > 16 ? 12 * L : 16));
    while (rows - 6 >= rmin && gx * ((ny + rows - 1) / rows) < want) rows -= 6;
    if (rows > ny) rows = ny;
    long gy = (ny + rows - 1) / rows;
    if (gx * gy > kMaxBlocks) {
        const long max_gy = kMaxBlocks / gx;
        rows = (ny + max_gy - 1) / max_gy;
        gy = (ny + rows - 1) / rows;
    }
    g->nx = nx; g->ny = ny; g->rows = (int)rows;
    g->row_lo = 0; g->row_hi = ny;
    *grid = dim3((unsigned)gx, (unsigned)gy);
    return true;
}

// red_src: which of the kernel's reductions the post functor consumes (it reads S_RED[0])
template <class C, class Post>
inline int launch_chain(Ctx *c, const kl_operator_t *op, C f, int nx, int ny, const Post &post, int red_src = 0) {
    constexpr int L = C::L;
    using D = ChainDims<L, C::VAROP>;
    using RG = ChainRing<C>;
    ChainGeo g;
    dim3 grid;
    if (!chain_geometry<L, C::VAROP>(c, nx, ny, &g, &grid, C::NIN == 1))
        return c->fail(KL_ERR_UNSUPPORTED, "grid too wide for the reduction buffer");
    // lines of the neighbour ranks are unknowns too (recomputed redundantly level by level)
    if (f.lo[0]) g.row_lo = -L;
    if (f.hi[0]) g.row_hi = ny + L;
    f.coef = op_coef(op);
    RedCtl rc = redctl(c);
    TMaps<C::NIN> tm;
    for (int a = 0; a < C::NIN; ++a) KL_TRY(tmap_encode_box(c, &tm.m[a], f.in[a], nx, ny, D::BWP, RG::SR));
    constexpr size_t smem = RG::bytes;
#define KL_CH_LAUNCH1(OPK, MG)                                                                         \
    {                                                                                                  \
        static bool attr[kMaxDevices] = {};   /* the shared-memory opt-in is per device */             \
        if (!attr[c->device % kMaxDevices]) {                                                          \
            cudaFuncSetAttribute(k_chain_tma<C, OPK, MG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            attr[c->device % kMaxDevices] = true;                                                      \
        }                                                                                              \
        k_chain_tma<C, OPK, MG><<<grid, kChainThreads, smem, c->stream>>>(f, g, rc, tm);               \
    }
#define KL_CH_LAUNCH(OPK)                                                                              \
    if constexpr (C::SINGLE_GPU) KL_CH_LAUNCH1(OPK, false)                                             \
    else if (f.lo[0] || f.hi[0]) KL_CH_LAUNCH1(OPK, true) else KL_CH_LAUNCH1(OPK, false)
    if (C::SINGLE_GPU && (f.lo[0] || f.hi[0])) return c->fail(KL_ERR_UNSUPPORTED, "launch_chain: single-GPU chain");
    if constexpr (C::VAROP) {
        if (op->kind != KL_OP_ANISO5_VAR || f.lo[0] || f.hi[0])
            return c->fail(KL_ERR_INVALID, "launch_chain: variable-coefficient chain on another operator");
        KL_CH_LAUNCH1(KL_OP_ANISO5_VAR, false)
    } else {
        switch (op->kind) {
            case KL_OP_POISSON5: KL_CH_LAUNCH(KL_OP_POISSON5) break;
            case KL_OP_ANISO5: KL_CH_LAUNCH(KL_OP_ANISO5) break;
            case KL_OP_STENCIL5:   // one GPU (prob_init): no multi-GPU instantiation
                if (f.lo[0] || f.hi[0]) return c->fail(KL_ERR_UNSUPPORTED, "launch_chain: KL_OP_STENCIL5 is single-GPU");
                KL_CH_LAUNCH1(KL_OP_STENCIL5, false)
                break;
            default: return c->fail(KL_ERR_INVALID, "launch_chain: not a built-in operator");
        }
    }
#undef KL_CH_LAUNCH
#undef KL_CH_LAUNCH1
    c->stats.kernel_launches++;
    // the post functor (scalar recurrences on the reduced sums) runs in its own one-warp kernel: the chain
    // kernels are not templated on it (each instantiation is 6 phases x L levels of code)
    const PostAny pa = to_any(post);
    if (C::NRED > 0 && pa.kind != PK_NoPost) {
        if (c->nranks > 1) return finish_reduction(c, C::NRED, pa, f.flags, f.step, f.run_on_conv, red_src);
        k_post<<<1, 32, 0, c->stream>>>(pa, f.flags, f.step, f.run_on_conv, c->d_S + S_RED, red_src);
        c->stats.kernel_launches++;
    }
    return KL_OK;
}

// ---------------------------------------------------------------------------
// degree-L Chebyshev preconditioner in one pass (oracle/krylov_extras.c ko_cheb, Saad Alg. 12.1):
//   level 0: u = r/theta, d = u ;  level l: d = fma(c1[l], d, c2[l]*(r - A u)) ; u = u + d ;  z = u_L
// Same arithmetic per point as FChebStep (kl_ops.cuh) => bit-identical results.
// mode 0: no reduction ; 1: acc0 = sum z*z ; 2: acc0 = sum r*z
// ---------------------------------------------------------------------------
// Reductions: acc0 = sum z*z and acc1 = sum r*z are BOTH kept (two DFMA per point instead of two DFMA and four
// selects on a run-time mode); the launcher tells the post functor which one to read (launch_chain red_src).
template <int L_>
struct ChCheb : ChainBase<1, L_, 1, 2> {
    double *z, *d_out;     // d_out != nullptr: also store d_L (continuation with FChebStep for degrees > kChainMaxL)
    int mode;              // 0: the sums are not used ; 1: z.z ; 2: r.z   (host side only)
    double theta;
    double c1[L_], c2[L_];
    FastDiv fd;
    __device__ __forceinline__ void init() { fd.set(theta); }
    __device__ __forceinline__ void level0(bool, size_t, const double (&raw)[1][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
        fd.div2(raw[0][0], raw[0][1], u[0], u[1]);
        cc[0][0] = u[0];
        cc[0][1] = u[1];
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW raw, const double (&)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *acc) const {
        const double2 rr = raw(0);
        const double r2[2] = {rr.x, rr.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double d = fma(c1[lv - 1], cin[0][e], c2[lv - 1] * (r2[e] - au[e]));
            u[e] = up[e] + d;
            cout[0][e] = d;
        }
        if (lv == L_ && out) {
            stg2(z + idx, u[0], u[1]);
            if (d_out) stg2(d_out + idx, cout[0][0], cout[0][1]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                acc[0] = fma(u[e], u[e], acc[0]);
                acc[1] = fma(r2[e], u[e], acc[1]);
            }
        }
    }
};

// Continuation chunk for degrees 7..12: steps s0+1 .. s0+L from the stored iterate and direction.
//   in[0] = z_{s0}, in[1] = d_{s0}, in[2] = r ;  level 0: u = z, d = d ;  level l as above ;  z = u_L
// z and d are read with the CTA's halo lines, so the outputs must be other buffers than the inputs.
template <int L_>
struct ChChebCont : ChainBase<3, L_, 1, 2> {
    static constexpr int SR = 2, NST = 6;                 // 12-line ring: keeps up to 6 lines behind the march
    static constexpr int MINB = L_ <= 4 ? 3 : 2;          // 74 KB of ring per CTA: 3 CTAs per SM at most
    double *z;
    int mode;
    double c1[L_], c2[L_];
    __device__ __forceinline__ void init() {}
    __device__ __forceinline__ void level0(bool, size_t, const double (&raw)[3][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            u[e] = raw[0][e];
            cc[0][e] = raw[1][e];
        }
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW raw, const double (&)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *acc) const {
        const double2 rr = raw(2);
        const double r2[2] = {rr.x, rr.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double d = fma(c1[lv - 1], cin[0][e], c2[lv - 1] * (r2[e] - au[e]));
            u[e] = up[e] + d;
            cout[0][e] = d;
        }
        if (lv == L_ && out) {
            stg2(z + idx, u[0], u[1]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                acc[0] = fma(u[e], u[e], acc[0]);
                acc[1] = fma(r2[e], u[e], acc[1]);
            }
        }
    }
};

// ---------------------------------------------------------------------------
// degree-L Jacobi-scaled Chebyshev on KL_OP_ANISO5_VAR in one pass (definition: tests/jacobi_cheb_twin.c):
//   level 0: u = (r*dinv)/theta, d = u ;  level l: d = fma(c1[l], d, c2[l]*((r - A u)*dinv)) ; u = u + d ;  z = u_L
// dinv = RN(1/diag) with the diagonal the kernel hands over.  Same arithmetic per point as k_jacobi_cheb_step
// (kl_ops.cu).  in = {r, kx, ky}: 24n B in, 8n B out (16n with d_out).  Reductions as ChCheb.
// ---------------------------------------------------------------------------
template <int L_>
struct ChJacCheb : ChainBase<3, L_, 1, 2> {
    static constexpr bool VAROP = true;
    static constexpr int SR = 2, NST = 6;       // 12-line ring: keeps up to L + 2 lines behind the march
    static constexpr int MINB = L_ <= 4 ? 3 : 2;   // 60-74 KB of ring per CTA: 3 CTAs per SM at most; L = 5, 6 spill under
                                                    // the 168-register cap of 3
    double *z, *d_out;     // d_out != nullptr: also store d_L (continuation with k_jacobi_cheb_step beyond kChainMaxL)
    int mode;              // 0: the sums are not used ; 1: z.z ; 2: r.z   (host side only)
    double theta;
    double c1[L_], c2[L_];
    FastDiv fd;
    __device__ __forceinline__ void init() { fd.set(theta); }
    __device__ __forceinline__ void level0(bool, size_t, const double (&raw)[3][2], const double (&dg)[2],
                                           double (&u)[2], double (&cc)[1][2], double *) const {
        fd.div2(raw[0][0] * __drcp_rn(dg[0]), raw[0][1] * __drcp_rn(dg[1]), u[0], u[1]);
        cc[0][0] = u[0];
        cc[0][1] = u[1];
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&dg)[2], const double (&cin)[1][2], RAW raw,
                                          const double (&)[1][2], double (&u)[2], double (&cout)[1][2],
                                          double *acc) const {
        const double2 rr = raw(0);
        const double r2[2] = {rr.x, rr.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double d = fma(c1[lv - 1], cin[0][e], c2[lv - 1] * ((r2[e] - au[e]) * __drcp_rn(dg[e])));
            u[e] = up[e] + d;
            cout[0][e] = d;
        }
        if (lv == L_ && out) {
            stg2(z + idx, u[0], u[1]);
            if (d_out) stg2(d_out + idx, cout[0][0], cout[0][1]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                acc[0] = fma(u[e], u[e], acc[0]);
                acc[1] = fma(r2[e], u[e], acc[1]);
            }
        }
    }
};

}  // namespace kl
