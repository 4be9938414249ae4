// kl_gmres.cu -- restarted, left-preconditioned GMRES(m) with Gram-Schmidt
// orthogonalisation applied twice.
//
// Reference: src/gmres_mgsr.f90  gmres_mgsr_omp :277-421, gmres_mgsr_mf :98-199.
//
// Data layout in HBM: the Krylov basis V is n x (m+1) column-major with leading
// dimension ldv >= n (each basis vector contiguous, 256-byte aligned); H is
// (m+1) x m column-major; g, cs, sn, y, final_err are small device arrays.
//
// One Arnoldi step (fused path):
//   stencil      V_j = w/h_val ; z = A V_j          (FScaleApply, 24n B)
//   stencil      w = cbpr2(z)                        (FCbpr2, 16n B)
//   k_vtw        h1 = V(:,0..j)^T w                  (8n(j+1) + 8n B)     |
//   k_wmvh       w -= V h1                           (8n(j+1) + 16n B)    | CGS2
//   k_vtw        h2 = V^T w ; H(:,j) = h1 + h2       (8n(j+1) + 8n B)     |
//   k_wmvh       w -= V h2 ; ||w||^2 ; Givens        (8n(j+1) + 16n B)    |
// or, with KL_ORTHO_MGS2, the reference's 2(j+1) sequential dot/axpy pairs
// (k_mgs_step: axpy with the previous column fused with the dot of the next).
// The Givens update, the residual estimate, n_out, the convergence flag and the
// residual history are produced on the device by one warp (givens_update_warp);
// the host reads them once per restart cycle.
#include <math.h>
#include <string.h>

#include <algorithm>

#include <cooperative_groups.h>

#include "kl_gmres.cuh"
#include "kl_tallskinny_tma.cuh"

namespace kl {

__global__ void k_givens(const GmresDev G, const int j, const int honor_skip = 0) {
    extern __shared__ double sm[];
    if (G.I[I_CONV_AT] >= 0) return;
    if (honor_skip && G.I[I_SKIP3]) return;
    givens_update_warp(G, j, sqrt(G.S[S_RED]), threadIdx.x, sm);
}

// Selective reorthogonalisation (KL_ORTHO_CGS2_SELECTIVE).  After  w' = w - V h1 ,  h2 = V^T w'  with
// ww = ||w||^2 (h1[nc]) and ww1 = ||w'||^2 (h2[nc]): if ||w'|| >= eta ||w|| the first pass lost at most
// a factor 1/eta of accuracy and the second update is skipped (h2 is discarded, ||w'|| is the new
// sub-diagonal); otherwise H(:,j) += h2 and the second update pass runs.  One warp, replicated on every rank.
__global__ void k_select(const GmresDev G, const double *h1, const double *h2, const int j, const int nc,
                         const double eta2) {
    extern __shared__ double sm[];
    if (G.I[I_CONV_AT] >= 0) return;
    const double ww = h1[nc], ww1 = h2[nc];
    const bool skip = ww1 >= eta2 * ww;
    if (skip) {
        if (threadIdx.x == 0) {
            G.I[I_SKIP3] = 1;
            G.I[I_NSKIP] = G.I[I_NSKIP] + 1;
            G.I[I_NSKIPCOLS] = G.I[I_NSKIPCOLS] + nc;
        }
        givens_update_warp(G, j, sqrt(ww1), threadIdx.x, sm);
    } else {
        double *Hj = G.H + (size_t)j * G.ldh;
        for (int c = threadIdx.x; c < nc; c += 32) Hj[c] = Hj[c] + h2[c];
        if (threadIdx.x == 0) G.I[I_SKIP3] = 0;
    }
}

// H(0..ncols-1, j) (+)= hvec   (gmres_mgsr.f90:351-353)
__global__ void k_hacc(const GmresDev G, const double *hv, const int j, const int ncols, const int accumulate) {
    if (G.I[I_CONV_AT] >= 0) return;
    double *Hj = G.H + (size_t)j * G.ldh;
    for (int c = threadIdx.x; c < ncols; c += blockDim.x)
        Hj[c] = accumulate ? Hj[c] + hv[c] : hv[c];
}

// ---- tall-skinny projection  out[c] = V(:,c) . w , c < ncols ------------------
// 8 warps per block arranged as RG row groups x CG column groups.  A warp keeps
// up to kTsCpw accumulators and streams its columns; w is read once per block
// trip (L1-shared between the column-group warps).  Deterministic two-stage
// reduction: block partials [col][block] -> last block sums over blocks.
template <int VEC>
__global__ void __launch_bounds__(kTsThreads, 2)
k_vtw(const double *__restrict__ V, const size_t ldv, const double *__restrict__ w, const size_t n,
      const int ncols, double *__restrict__ partials, unsigned int *counter, double *__restrict__ out,
      const GmresDev G, const int j, const int h_mode /* 0: none, 1: H=out, 2: H+=out */,
      const int *__restrict__ flags) {
    if (flags && flags[I_CONV_AT] >= 0) return;
    __shared__ double s_part[kTsWarps][kTsCpw];
    __shared__ int s_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int ncg = (ncols + kTsCpw - 1) / kTsCpw;
    int CG = 1;
    while (CG < ncg && CG < kTsWarps) CG <<= 1;
    const int RG = kTsWarps / CG;
    const int cg = wid % CG, rg = wid / CG;
    constexpr size_t WROWS = (size_t)32 * kTsU * VEC;   // rows per warp trip
    const size_t TR = WROWS * RG;                       // rows per block trip
    const int cols_per_pass = CG * kTsCpw;
    for (int cbase = 0; cbase < ncols; cbase += cols_per_pass) {
        const int c0 = cbase + cg * kTsCpw;
        double acc[kTsCpw];
#pragma unroll
        for (int c = 0; c < kTsCpw; ++c) acc[c] = 0.0;
        for (size_t t0 = (size_t)blockIdx.x * TR; t0 < n; t0 += (size_t)gridDim.x * TR) {
            const size_t r0 = t0 + (size_t)rg * WROWS + (size_t)lane * VEC;
            double wv[kTsU][VEC];
#pragma unroll
            for (int u = 0; u < kTsU; ++u) {
                const size_t r = r0 + (size_t)u * 32 * VEC;
                if (r < n) {
                    if (VEC == 2) {
                        double2 t = ldg2(w + r);
                        wv[u][0] = t.x; wv[u][VEC - 1] = t.y;
                    } else {
                        wv[u][0] = __ldg(w + r);
                    }
                } else {
                    wv[u][0] = 0.0; wv[u][VEC - 1] = 0.0;
                }
            }
#pragma unroll
            for (int c = 0; c < kTsCpw; ++c) {
                if (c0 + c < ncols) {
                    const double *col = V + (size_t)(c0 + c) * ldv;
#pragma unroll
                    for (int u = 0; u < kTsU; ++u) {
                        const size_t r = r0 + (size_t)u * 32 * VEC;
                        if (r < n) {
                            if (VEC == 2) {
                                double2 t = ldg2(col + r);
                                acc[c] = fma(t.x, wv[u][0], acc[c]);
                                acc[c] = fma(t.y, wv[u][VEC - 1], acc[c]);
                            } else {
                                acc[c] = fma(__ldg(col + r), wv[u][0], acc[c]);
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int c = 0; c < kTsCpw; ++c) {
            double s = warp_sum(acc[c]);
            if (lane == 0) s_part[wid][c] = s;
        }
        __syncthreads();
        if (threadIdx.x < cols_per_pass) {
            const int col = cbase + threadIdx.x;
            if (col < ncols) {
                const int g = threadIdx.x / kTsCpw, c = threadIdx.x % kTsCpw;
                double s = 0.0;
                for (int r = 0; r < RG; ++r) s += s_part[r * CG + g][c];
                partials[(size_t)col * kTsMaxBlocks + blockIdx.x] = s;
            }
        }
        __syncthreads();
    }
    // ---- grid stage
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned prev = atomicAdd(counter, 1u);
        s_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int col = wid; col < ncols; col += kTsWarps) {
        const volatile double *p = partials + (size_t)col * kTsMaxBlocks;
        double s = 0.0;
        for (unsigned b = lane; b < gridDim.x; b += 32) s += p[b];
        s = warp_sum(s);
        if (lane == 0) {
            out[col] = s;
            if (h_mode) {
                double *Hj = G.H + (size_t)j * G.ldh;
                Hj[col] = (h_mode == 2) ? Hj[col] + s : s;
            }
        }
    }
    if (threadIdx.x == 0) *counter = 0u;
}

// ---- w_out = w - V(:,0..ncols-1) h  (+ ||w_out||^2, + Givens in the last block) --
// FMA order = column order (the CPU twin's CGS2 loop).  wmvh_pass is the body (whole grid); k_wmvh the kernel.
template <int VEC>
__device__ __forceinline__ void wmvh_pass(const double *__restrict__ V, const size_t ldv, double *w, const size_t n,
                                          const int ncols, const double *__restrict__ h, const RedCtl &rc,
                                          const int want_norm, const GmresDev &G, const int j, const int fuse_givens,
                                          double *sm /* max(ncols, 3*(m+2)) doubles */) {
    double *sh = sm;
    for (int c = threadIdx.x; c < ncols; c += kTsThreads) sh[c] = h[c];
    __syncthreads();
    double nacc = 0.0;
    const size_t nchunk = n / VEC;
    for (size_t ch = (size_t)blockIdx.x * kTsThreads + threadIdx.x; ch < nchunk;
         ch += (size_t)gridDim.x * kTsThreads) {
        const size_t r = ch * VEC;
        double a[VEC];
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(w + r);
            a[0] = t.x; a[VEC - 1] = t.y;
        } else {
            a[0] = w[r];
        }
        int c = 0;
        for (; c + 8 <= ncols; c += 8) {
            double v[8][VEC];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double *col = V + (size_t)(c + q) * ldv + r;
                if (VEC == 2) {
                    double2 t = ldg2(col);
                    v[q][0] = t.x; v[q][VEC - 1] = t.y;
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
        for (; c < ncols; ++c) {
            const double *col = V + (size_t)c * ldv + r;
            const double hq = -sh[c];
            if (VEC == 2) {
                double2 t = ldg2(col);
                a[0] = fma(hq, t.x, a[0]);
                a[VEC - 1] = fma(hq, t.y, a[VEC - 1]);
            } else {
                a[0] = fma(hq, __ldg(col), a[0]);
            }
        }
        if (VEC == 2) stg2(w + r, a[0], a[VEC - 1]);
        else w[r] = a[0];
#pragma unroll
        for (int e = 0; e < VEC; ++e) nacc = fma(a[e], a[e], nacc);
    }
    if (!(want_norm & 1)) return;
    __syncthreads();
    __shared__ double s_red[kTsWarps];
    __shared__ int s_flag;
    double accv[1] = {nacc};
    block_sum<1, kTsThreads>(accv, s_red);
    if (grid_sum<1, kTsThreads>(accv, rc, gridDim.x, blockIdx.x, &s_flag, s_red)) {
        if (fuse_givens && threadIdx.x < 32) givens_update_warp(G, j, sqrt(rc.red[0]), threadIdx.x, sm);
    }
}

template <int VEC>
__global__ void __launch_bounds__(kTsThreads)
k_wmvh(const double *__restrict__ V, const size_t ldv, double *w, const size_t n, const int ncols,
       const double *__restrict__ h, const RedCtl rc, const int want_norm, const GmresDev G,
       const int j, const int fuse_givens, const int *__restrict__ flags) {
    // want_norm: bit 0 = reduce ||w||^2 ; bit 1 = selective mode: do nothing when I_SKIP3 is set
    griddep_wait();
    griddep_launch();
    if (flags && flags[I_CONV_AT] >= 0) return;
    if ((want_norm & 2) && flags[I_SKIP3]) return;
    extern __shared__ double sm[];   // max(ncols, 3*(m+2)) doubles + reduction scratch
    wmvh_pass<VEC>(V, ldv, w, n, ncols, h, rc, want_norm, G, j, fuse_givens, sm);
}

// ---- the whole CGS2 orthogonalisation of one Arnoldi step as ONE cooperative kernel (single GPU, small grids) ----
//   h1 = V^T w ; H(:,j) = h1      | grid barrier |  w -= V h1 ; h2 = V^T w ; H(:,j) += h2   | grid barrier |
//   w -= V h2 ; ||w|| ; Givens, residual estimate, convergence flag (last block)
// At 300^2 (BASELINE config 1, the reference's own headline problem) V is L2-resident and each of the three passes is
// a 15-20 us kernel whose time is launch, ramp and reduction tail, not data; as three phases of one persistent
// kernel they cost one launch and two ~2 us barriers.  Same device code, same partial-sum order => same bits.
__global__ void __launch_bounds__(kTsThreads, 2)
k_cgs2_coop(const __grid_constant__ CUtensorMap tmV, const double *__restrict__ V, const size_t ldv, double *w,
            const size_t n, const int nc, const int RM, double *__restrict__ partials, unsigned int *counter,
            const RedCtl rc, const GmresDev G, const int j, const int *__restrict__ flags, unsigned int *sync_flag) {
    if (flags && flags[I_CONV_AT] >= 0) return;          // grid-uniform: every CTA leaves before the first barrier
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // Grid barriers without cooperative_groups: a pass already ends with "every CTA arrives at a counter, the last one
    // sums the partials"; the other CTAs only have to wait for that block's result, so the barrier is the arrival
    // plus one release / acquire flag (its value read here, before any CTA can have arrived anywhere, + the pass
    // number).  The cooperative launch is kept for its co-residency guarantee.
    unsigned f0;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(f0) : "l"(sync_flag) : "memory");
    const TsTail none{nullptr, nullptr, 0};
    ts_pass<false>(tmV, w, n, nc, RM, nullptr, partials, counter, G.hvec, G, j, 1, -1, none, smem_raw, sync_flag, f0 + 1u);
    ts_pass<true>(tmV, w, n, nc, RM, G.hvec, partials, counter, G.hvec2, G, j, 2, -1, none, smem_raw, sync_flag, f0 + 2u);
    wmvh_pass<2>(V, ldv, w, n, nc, G.hvec2, rc, 1, G, j, 1, reinterpret_cast<double *>(smem_raw));
}

// ---- one Arnoldi step's operator part in ONE pass (temporally blocked, kl_chain_tma.cuh) -----------------------
//   V_j = w / h ; z = A V_j ; w' = cbpr2(z) = z/d + alpha (z - A (z/d))     gmres_mgsr.f90:384,336,337 ; chebyshev.f90:27-37
// reads w, writes V_j and w': 24n B and one launch instead of 24n + 16n B and two (FScaleApply, FCbpr2).  Same
// arithmetic per point as those two kernels (same divisions, same fma), so the results are bit-identical.
struct ChGmresStep : ChainBase<1, 2, 1, 0> {
    double *v_out, *w_out;
    const double *S;
    int s_idx;
    double d, calpha;
    FastDiv fh, fd;
    __device__ __forceinline__ void init() {
        fh.set(S[s_idx]);
        fd.set(d);
    }
    __device__ __forceinline__ void level0(bool out, size_t idx, const double (&raw)[1][2], double (&u)[2],
                                           double (&cc)[1][2], double *) const {
        fh.div2(raw[0][0], raw[0][1], u[0], u[1]);                                   // :384
        cc[0][0] = cc[0][1] = 0.0;
        if (out) stg2(v_out + idx, u[0], u[1]);
    }
    template <class RAW>
    __device__ __forceinline__ void level(int lv, bool out, size_t idx, const double (&up)[2], const double (&au)[2],
                                          const double (&cin)[1][2], RAW, const double (&)[1][2], double (&u)[2],
                                          double (&cout)[1][2], double *) const {
        if (lv == 1) {
            fd.div2(au[0], au[1], u[0], u[1]);                                       // chebyshev.f90:28-30  z0 = r/d, r = A V_j
            cout[0][0] = au[0];
            cout[0][1] = au[1];
        } else {
            u[0] = fma(calpha, cin[0][0] - au[0], up[0]);                            // :34-36
            u[1] = fma(calpha, cin[0][1] - au[1], up[1]);
            cout[0][0] = cout[0][1] = 0.0;
            if (out) stg2(w_out + idx, u[0], u[1]);
        }
    }
};

// ---- back substitution by one warp (gmres_mgsr.f90:394-398) -------------------
// lane 0 runs the reference's sequential recurrence; the warp stages row i of H.
__global__ void k_backsolve(const GmresDev G) {
    extern __shared__ double sm[];   // m doubles row + m doubles y
    const int lane = threadIdx.x;
    const int n_out = G.I[I_NOUT];
    double *row = sm, *ys = sm + G.m;
    for (int i = lane; i < G.m; i += 32) ys[i] = 0.0;
    __syncwarp();
    for (int i = n_out - 1; i >= 0; --i) {
        for (int k = i + lane; k < n_out; k += 32) row[k] = G.H[(size_t)k * G.ldh + i];
        __syncwarp();
        if (lane == 0) {
            double s = 0.0;
            for (int k = i + 1; k < n_out; ++k) s = fma(row[k], ys[k], s);
            ys[i] = (G.g[i] - s) / row[i];
        }
        __syncwarp();
    }
    for (int i = lane; i < G.m; i += 32) G.y[i] = ys[i];
}

// ---- x += V(:,0..n_out-1) y   (gmres_mgsr.f90:400-406) -------------------------
template <int VEC>
__global__ void __launch_bounds__(kTsThreads)
k_xpvy(const double *__restrict__ V, const size_t ldv, double *x, const size_t n, const GmresDev G) {
    extern __shared__ double sy[];
    const int n_out = G.I[I_NOUT];
    for (int c = threadIdx.x; c < n_out; c += kTsThreads) sy[c] = G.y[c];
    __syncthreads();
    const size_t nchunk = n / VEC;
    for (size_t ch = (size_t)blockIdx.x * kTsThreads + threadIdx.x; ch < nchunk;
         ch += (size_t)gridDim.x * kTsThreads) {
        const size_t r = ch * VEC;
        double s[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) s[e] = 0.0;
        int c = 0;
        for (; c + 8 <= n_out; c += 8) {
            double v[8][VEC];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double *col = V + (size_t)(c + q) * ldv + r;
                if (VEC == 2) {
                    double2 t = ldg2(col);
                    v[q][0] = t.x; v[q][VEC - 1] = t.y;
                } else {
                    v[q][0] = __ldg(col);
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
#pragma unroll
                for (int e = 0; e < VEC; ++e) s[e] = fma(v[q][e], sy[c + q], s[e]);
        }
        for (; c < n_out; ++c) {
            const double *col = V + (size_t)c * ldv + r;
            if (VEC == 2) {
                double2 t = ldg2(col);
                s[0] = fma(t.x, sy[c], s[0]);
                s[VEC - 1] = fma(t.y, sy[c], s[VEC - 1]);
            } else {
                s[0] = fma(__ldg(col), sy[c], s[0]);
            }
        }
        if (VEC == 2) {
            double2 t = *reinterpret_cast<const double2 *>(x + r);
            stg2(x + r, t.x + s[0], t.y + s[VEC - 1]);
        } else {
            x[r] = x[r] + s[0];
        }
    }
}

static inline int ts_grid(size_t n, int vec) {
    size_t rows_per_block = (size_t)32 * kTsU * vec;  // at least one warp trip
    size_t b = (n + rows_per_block - 1) / rows_per_block;
    size_t cap = (size_t)kNumSM * 2;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}
static inline int upd_grid(size_t nchunk) {
    size_t b = (nchunk + kTsThreads - 1) / kTsThreads;
    size_t cap = (size_t)kNumSM * 8;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

int launch_vtw(Ctx *c, const double *V, size_t ldv, const double *w, size_t n, int ncols, double *out,
               const GmresDev &G, int j, int h_mode, bool gated) {
    const int vec = (n % 2 == 0 && ldv % 2 == 0) ? 2 : 1;
    const int grid = ts_grid(n, vec);
    const int hm = c->nranks == 1 ? h_mode : 0;
    if (vec == 2)
        k_vtw<2><<<grid, kTsThreads, 0, c->stream>>>(V, ldv, w, n, ncols, c->d_partials, c->d_counter + 1,
                                                     out, G, j, hm, gated ? c->d_I : nullptr);
    else
        k_vtw<1><<<grid, kTsThreads, 0, c->stream>>>(V, ldv, w, n, ncols, c->d_partials, c->d_counter + 1,
                                                     out, G, j, hm, gated ? c->d_I : nullptr);
    c->stats.kernel_launches++;
    if (c->nranks > 1) {
        KL_TRY(comm_allreduce(c, out, ncols));
        if (h_mode) {
            k_hacc<<<1, 128, 0, c->stream>>>(G, out, j, ncols, h_mode == 2);
            c->stats.kernel_launches++;
        }
    }
    return KL_OK;
}

// Can the TMA tall-skinny kernels run?  EVERY rank must take the same decision (the two paths all-reduce different
// numbers of values and only one of them can skip the second pass), so on several ranks it is taken from the global
// grid and the smallest / largest slab of the partition, never from this rank's own n.
bool ts_tma_ok(Ctx *c, size_t n, size_t ldv, int nc, int nx, int ny) {
    if (!(c->opt_tma && nc >= 1 && nc <= kTsWarps * kTsCpw && ldv % 2 == 0)) return false;
    if (c->nranks == 1 || nx <= 0) return n % 2 == 0 && n >= 4096 && n < (size_t)1 << 31;
    const size_t n_min = (size_t)nx * (size_t)(ny / c->nranks), n_max = (size_t)nx * (size_t)((ny + c->nranks - 1) / c->nranks);
    return nx % 2 == 0 && n_min >= 4096 && n_max < (size_t)1 << 31;
}

int launch_ts_tma(Ctx *c, bool update, const double *V, size_t ldv, int ncols_total, double *w, size_t n, int nc,
                  const double *h_in, double *out, const GmresDev &G, int j, int h_mode, bool gated,
                  long long tail0, const double *tail_T, double *tail_tvec, int tail_ldt) {
    const TsTail tt{tail_T, tail_tvec, tail_ldt};
    CUtensorMap tm;
    KL_TRY(tmap_encode_v(c, &tm, V, n, ldv, ncols_total, nc));
    const size_t smem = ts_tma_smem(nc);
    static bool attr_done[kMaxDevices] = {};   // the shared-memory opt-in is per device
    if (!attr_done[c->device % kMaxDevices]) {
        cudaFuncSetAttribute(k_ts_tma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024);
        cudaFuncSetAttribute(k_ts_tma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024);
        attr_done[c->device % kMaxDevices] = true;
    }
    const int RM = ts_rm(nc);
    size_t ntiles = (n + (size_t)kTsRB * RM - 1) / ((size_t)kTsRB * RM);
    int grid = (int)std::min<size_t>(ntiles, (size_t)kNumSM * 2);
    if (c->opt_ts_blocks > 0 && c->opt_ts_blocks < grid) grid = c->opt_ts_blocks;
    const int hm = c->nranks == 1 ? h_mode : 0;
    const int *fl = gated ? c->d_I : nullptr;
    if (update)
        KL_CUDA(c, launch_k(c, false, k_ts_tma<true>, dim3(grid), dim3(kTsThreads), smem, tm, w, n, nc, RM, h_in,
                            c->d_partials, c->d_counter + 1, out, G, j, hm, fl, tail0, tt));
    else
        KL_CUDA(c, launch_k(c, false, k_ts_tma<false>, dim3(grid), dim3(kTsThreads), smem, tm, w, n, nc, RM, h_in,
                            c->d_partials, c->d_counter + 1, out, G, j, hm, fl, tail0, tt));
    c->stats.kernel_launches++;
    if (c->nranks > 1) {
        KL_TRY(comm_allreduce(c, out, nc + (tail0 >= 0 ? 1 : 0)));
        if (h_mode) {
            k_hacc<<<1, 128, 0, c->stream>>>(G, out, j, nc, h_mode == 2);
            c->stats.kernel_launches++;
        }
    }
    return KL_OK;
}

#ifdef KL_TRACE
extern "C" int kl_debug_trace_ts(unsigned long long *out, int n) {
    return cudaMemcpyFromSymbol(out, g_trace_ts, sizeof(unsigned long long) * n) == cudaSuccess ? 0 : -1;
}
#endif

// cooperative CGS2 step (see k_cgs2_coop): single GPU, TMA path, problems small enough to be launch-bound
bool cgs2_coop_ok(Ctx *c, size_t n, size_t ldv, int m) {
    return c->nranks == 1 && c->opt_coop && !c->opt_profile && c->opt_ortho == KL_ORTHO_CGS2 &&
           ts_tma_ok(c, n, ldv, m + 1) && n <= ((size_t)1 << 21);
}
int launch_cgs2_coop(Ctx *c, const double *V, size_t ldv, int ncols_total, double *w, size_t n, int nc,
                     const GmresDev &G, int j) {
    CUtensorMap tm;
    KL_TRY(tmap_encode_v(c, &tm, V, n, ldv, ncols_total, nc));
    const size_t smem = std::max(ts_tma_smem(nc), sizeof(double) * (size_t)std::max(nc + 8, 3 * (G.m + 2)) + 256);
    static bool attr_done[kMaxDevices] = {};
    if (!attr_done[c->device % kMaxDevices]) {
        cudaFuncSetAttribute(k_cgs2_coop, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024);
        attr_done[c->device % kMaxDevices] = true;
    }
    int RM = ts_rm(nc);
    const size_t ntiles = (n + (size_t)kTsRB * RM - 1) / ((size_t)kTsRB * RM);
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_cgs2_coop, kTsThreads, smem) != cudaSuccess || occ < 1)
        return c->fail(KL_ERR_CUDA, "k_cgs2_coop occupancy");
    int grid = (int)std::min<size_t>(ntiles, (size_t)kNumSM * std::min(occ, 2));
    RedCtl rc = redctl(c);
    const int *fl = c->d_I;
    const double *Vc = V;
    size_t ldv_ = ldv, n_ = n;
    unsigned int *counter = c->d_counter + 1;
    double *partials = c->d_partials;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kTsThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = c->stream;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    unsigned int *sync_flag = c->d_counter + 8;
    KL_CUDA(c, cudaLaunchKernelEx(&cfg, k_cgs2_coop, tm, Vc, ldv_, w, n_, nc, RM, partials, counter, rc, G, j, fl, sync_flag));
    c->stats.kernel_launches++;
    return KL_OK;
}

int launch_wmvh(Ctx *c, const double *V, size_t ldv, double *w, size_t n, int ncols, const double *h,
                bool want_norm, const GmresDev &G, int j, bool givens, bool gated, bool honor_skip = false) {
    const int vec = (n % 2 == 0 && ldv % 2 == 0) ? 2 : 1;
    const int grid = upd_grid(n / vec);
    const size_t smem = sizeof(double) * std::max(ncols + 8, 3 * (G.m + 2));
    const int fuse = (givens && c->nranks == 1) ? 1 : 0;
    const int wn = (want_norm ? 1 : 0) | (honor_skip ? 2 : 0);
    RedCtl rc = redctl(c);
    const int *fl = (gated || honor_skip) ? c->d_I : nullptr;
    if (vec == 2)
        KL_CUDA(c, launch_k(c, false, k_wmvh<2>, dim3(grid), dim3(kTsThreads), smem, V, ldv, w, n, ncols, h, rc, wn, G, j,
                            fuse, fl));
    else
        KL_CUDA(c, launch_k(c, false, k_wmvh<1>, dim3(grid), dim3(kTsThreads), smem, V, ldv, w, n, ncols, h, rc, wn, G, j,
                            fuse, fl));
    c->stats.kernel_launches++;
    if (want_norm && c->nranks > 1) {
        KL_TRY(comm_allreduce(c, c->d_S + S_RED, 1));
        if (givens) {
            k_givens<<<1, 32, sizeof(double) * 3 * (G.m + 2), c->stream>>>(G, j, honor_skip ? 1 : 0);
            c->stats.kernel_launches++;
        }
    }
    return KL_OK;
}

int launch_backsolve(Ctx *c, const GmresDev &G) {
    k_backsolve<<<1, 32, sizeof(double) * 2 * G.m, c->stream>>>(G);
    c->stats.kernel_launches++;
    return KL_OK;
}

// Gram-matrix epilogue shared with the Householder solver: G[c*(k)+i] = V_i . V_c, i <= c
int gram_lower(Ctx *c, const double *V, size_t ldv, size_t n, int k, double *d_gram, std::vector<double> &out) {
    GmresDev none{};
    for (int col = 0; col < k; ++col)
        KL_TRY(launch_vtw(c, V, ldv, V + (size_t)col * ldv, n, col + 1, d_gram + (size_t)col * k, none, 0, 0, false));
    out.assign((size_t)k * k, 0.0);
    KL_CUDA(c, cudaMemcpyAsync(out.data(), d_gram, sizeof(double) * k * k, cudaMemcpyDeviceToHost, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    return KL_OK;
}

int gmres_mgsr_solve(Ctx *c, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                            int m, double tol, double *final_err, double *v_err, int *n_out_p,
                            int *restart_out_p, const kl_precond_t *M, const double *params, int nparams,
                            int mf) {
    if (!c || !A || !b || !x || !final_err || !v_err || !n_out_p || !restart_out_p) return KL_ERR_INVALID;
    if (m < 1 || m + 1 > kMaxCols) return c->fail(KL_ERR_INVALID, "restart length m out of range");
    KL_TRY(x0_check(c, b, x));
    Prob P;
    KL_TRY(prob_init(&P, c, A, M, params, nparams, nx, ny));
    const bool prec = P.pc.kind != KL_PC_NONE;
    const bool fused = c->opt_fuse && P.builtin_op();
    const size_t n = P.n;
    const size_t ldv = (n + 31) & ~size_t(31);
    const int ldh = m + 1;
    const int vec = (n % 2 == 0) ? 2 : 1;
    c->stats = kl_stats_t{};
    prof_reset(c);
    const cudaEvent_t evA = c->ev2, evB = c->ev3;     // owned by the handle (no leak on the error paths)
    KL_CUDA(c, cudaEventRecord(evA, c->stream));

    const bool dev = c->pointer_mode == KL_POINTER_DEVICE;
    size_t need = ws_need(ldv * (size_t)(m + 1)) + 7 * ws_need(n) + ws_need((size_t)ldh * m) +
                  10 * ws_need(m + 2) + ws_need((size_t)(m + 2) * (m + 2));
    KL_TRY(ws_reserve(c, need));
    ws_reset(c);
    double *V = ws_take<double>(c, ldv * (size_t)(m + 1));
    double *w = ws_take<double>(c, n), *z = ws_take<double>(c, n), *aux = ws_take<double>(c, n);
    double *aux2 = ws_take<double>(c, n);
    double *w2 = ws_take<double>(c, n);     // second w buffer of the one-pass step (its input and output differ)
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
    G.hvec2 = ws_take<double>(c, m + 2);
    double *d_gram = ws_take<double>(c, (size_t)(m + 2) * (m + 2));
    G.S = c->d_S; G.I = c->d_I; G.hist = c->d_hist; G.hist_cap = c->hist_cap;
    G.m = m; G.ldh = ldh; G.mf = mf;

    if (!dev) KL_TRY(stage_in(c, db, b, n));
    if (c->opt_x0) KL_TRY(stage_in(c, dx, x, n));                               // x = x0 (KL_OPT_X0)
    else KL_CUDA(c, cudaMemsetAsync(dx, 0, n * sizeof(double), c->stream));     // x = 0 (:304)
    KL_CUDA(c, cudaMemsetAsync(G.fe, 0, (m + 2) * sizeof(double), c->stream));  // final_err = 0
    KL_CUDA(c, cudaMemsetAsync(c->d_I, 0, sizeof(int) * I_COUNT, c->stream));
    {
        double S0[32] = {0};
        S0[S_TOL] = tol;
        KL_CUDA(c, cudaMemcpyAsync(c->d_S, S0, sizeof S0, cudaMemcpyHostToDevice, c->stream));
        int m1 = -1;
        KL_CUDA(c, cudaMemcpyAsync(c->d_I + I_CONV_AT, &m1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    {   // beta0 = norm2(b) (:307)
        PDot2 d;
        set_gate(d, c, false);
        d.a = db; d.b = db; d.c = nullptr; d.d = nullptr;
        KL_TRY(launch_pointwise(c, d, n, PostStoreRed{c->d_S, S_BETA0, 1}));
    }
    if (c->opt_x0) {
        // the first cycle's beta = ||M^-1 (b - A x0)|| against the ||b|| that final_err is measured with: x0 that
        // already passes the test returns before a cycle (beta = 0 would make V_1 = w/0)
        KL_TRY(op_resid(&P, dx, db, z, false));
        if (prec) KL_TRY(pc_apply(&P, z, w, aux, aux2, 0, false, NoPost{}));
        double beta = 0.0;
        KL_TRY(x0_norm(c, prec ? w : z, n, &beta));
        if (beta == 0.0 || beta / c->h_pinned[S_BETA0] < tol) {
            KL_TRY(x0_zero_step(c));
            for (int i = 0; i < m; ++i) final_err[i] = 0.0;
            for (int i = 0; i <= m; ++i) v_err[i] = 0.0;
            *n_out_p = 0;
            *restart_out_p = 1;
            return KL_OK;
        }
    }
    KL_CUDA(c, cudaEventRecord(c->ev0, c->stream));

    const int max_restarts = c->opt_max_restarts;
    int status = KL_NOT_CONVERGED, n_out = 0, restart_out = max_restarts, cycles = 0;
    double bytes = 0.0;
    double *const w_base = w, *const z_base = z;
    // V_j = w/h, z = A V_j and w = cbpr2(z) as one temporally blocked pass (same decision on every rank)
    // (large grids only: the temporally blocked kernel's CTAs are 240 columns x 48 lines, which is 14 CTAs at 300^2 --
    // there the two small stencil kernels, 76 CTAs each, are faster: 57 vs 61 us per step measured)
    const bool chain_step = fused && P.pc.kind == KL_PC_CBPR2 && chain_ok(&P, 2) &&
                            ((size_t)P.nx * (size_t)(P.ny / c->nranks) >= (size_t)c->opt_chain_step_min ||
                             (c->nranks == 1 && (size_t)P.nx * (size_t)P.ny <= ((size_t)1 << 18)));   // launch-bound grids:
                            // one launch less per step (300^2: 48.9 -> 44.3 us with 6-line marches); in between the
                            // two stencil kernels fill the GPU better than the chain kernel's few CTAs
    const Cbpr2Coef cbc = chain_step ? cbpr2_coef(P.params) : Cbpr2Coef{1.0, 0.0};
    const bool coop = cgs2_coop_ok(c, n, ldv, m);
    // One restart cycle = a fixed sequence of launches (every pointer, column count and step index is known on
    // the host; convergence is a device-side gate), so it can be captured once and replayed as a CUDA graph:
    // at 300^2 (BASELINE config 1) a cycle is ~480 launches of 5-20 us kernels and launch overhead dominates.
    auto enqueue_cycle = [&]() -> int {
        const PdlScope pdl_scope(c, c->nranks == 1);     // programmatic dependent launch for the whole cycle
        w = w_base;
        z = z_base;
        double *wn = w2;
        // g = 0 ; H = 0 (:312).  (V = 0 is not needed: every column is written before it is read.)
        KL_CUDA(c, cudaMemsetAsync(G.H, 0, sizeof(double) * (size_t)ldh * m, c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.g, 0, sizeof(double) * (m + 2), c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.cs, 0, sizeof(double) * (m + 2), c->stream));
        KL_CUDA(c, cudaMemsetAsync(G.sn, 0, sizeof(double) * (m + 2), c->stream));
        // w = M^-1 (b - A x) ; beta = ||w|| ; g(1) = beta (:314-324)
        KL_TRY(op_resid(&P, dx, db, z, false));
        if (prec) {
            KL_TRY(pc_apply(&P, z, w, aux, aux2, 1, false, PostBeta{G}));
        } else {
            PDot2 d;
            set_gate(d, c, false);
            d.a = z; d.b = z; d.c = nullptr; d.d = nullptr;
            KL_TRY(launch_pointwise(c, d, n, PostBeta{G}));
            std::swap(w, z);
        }
        bytes += (24.0 + (prec ? 16.0 : 8.0)) * n;
        int norm_idx = S_NORM;  // norm of the vector in `w` that becomes V_j
        for (int j = 0; j < m; ++j) {
            double *Vj = V + (size_t)j * ldv;
            // V_j = w / norm ; z = A V_j   (:325-329 / :384 of the previous step ; :336).
            // omp: V_j is also written when the previous step converged (:384 precedes :385).
            if (chain_step) {
                ProfScope ps(c, 0, "gmres_scale_apply_precond (chain: V_j=w/h; z=A V_j; w=cbpr2(z))", 24.0 * n);
                Halo H;
                const double *vecs[1] = {w};
                KL_TRY(halo_exchange_lines(&P, vecs, 1, 2, &H));
                ChGmresStep f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true, j - 1, mf ? 0 : 1);
                f.v_out = Vj; f.w_out = wn; f.S = c->d_S; f.s_idx = norm_idx; f.d = cbc.d; f.calpha = cbc.alpha;
                KL_TRY(launch_chain(c, &P.op, f, P.nx, P.nyl, NoPost{}));
                std::swap(w, wn);
            } else if (fused) {
                ProfScope ps(c, 0, "gmres_scale_apply (stencil: V_j=w/h; z=A V_j)", 24.0 * n);
                Halo H;
                const double *vecs[1] = {w};
                KL_TRY(halo_exchange(&P, vecs, 1, &H));
                FScaleApply f;
                set_io(f, &P, vecs, H);
                set_gate(f, c, true, j - 1, mf ? 0 : 1);
                f.v_out = Vj; f.z = z; f.S = c->d_S; f.s_idx = norm_idx;
                KL_TRY(launch_stencil(c, &P.op, f, P.nx, P.nyl, NoPost{}));
            } else {
                PScale s;
                set_gate(s, c, true, j - 1, mf ? 0 : 1);
                s.in = w; s.out = Vj; s.S = c->d_S; s.s_idx = norm_idx;
                KL_TRY(launch_pointwise(c, s, n, NoPost{}));
                KL_TRY(op_apply(&P, Vj, z, true));
            }
            // w = M^-1 z (:337)
            if (chain_step) {
                // done above
            } else if (prec) {
                ProfScope ps(c, 1, "gmres_precond (stencil: w=M^-1 z)", 16.0 * n);
                KL_TRY(pc_apply(&P, z, w, aux, aux2, 0, true, NoPost{}));
            } else std::swap(w, z);
            double *wj = w;
            const int ncols = j + 1;
            if (c->opt_ortho == KL_ORTHO_MGS2) {
                // reference order: for k=1,2: for i=1..j: h = w.V_i ; H(i,j) += h ; w -= h V_i
                const int total = 2 * ncols;
                for (int t = 0; t <= total; ++t) {
                    PMgsStep s;
                    set_gate(s, c, true);
                    s.w = wj; s.S = c->d_S;
                    s.vprev = (t > 0) ? V + (size_t)((t - 1) % ncols) * ldv : nullptr;
                    s.vcur = (t < total) ? V + (size_t)(t % ncols) * ldv : nullptr;
                    s.want_norm = (t == total);
                    if (t < total) {
                        KL_TRY(launch_pointwise(c, s, n, PostMgs{G, j, t % ncols}));
                    } else {
                        // last axpy fused with ||w||^2 ; Givens after it
                        KL_TRY(launch_pointwise(c, s, n, NoPost{}));
                        k_givens<<<1, 32, sizeof(double) * 3 * (m + 2), c->stream>>>(G, j);
                        c->stats.kernel_launches++;
                    }
                }
                bytes += (32.0 * total + 24.0) * n;
            } else {
                if (c->opt_ortho == KL_ORTHO_CGS2_SELECTIVE && ts_tma_ok(c, n, ldv, ncols, P.nx, P.ny)) {
                    const double eta = c->opt_reorth_eta_permille * 1e-3;
                    { ProfScope ps(c, 2, "gmres_vtw_tma (h1=V^T w, TMA-staged tall-skinny projection)", (8.0 * ncols + 8.0) * n);
                      KL_TRY(launch_ts_tma(c, false, V, ldv, m + 1, wj, n, ncols, nullptr, G.hvec, G, j, 1, true, 0)); }
                    { ProfScope ps(c, 4, "gmres_wmvh_vtw_tma (w-=V h1 fused with h2=V^T w)", (8.0 * ncols + 16.0) * n);
                      KL_TRY(launch_ts_tma(c, true, V, ldv, m + 1, wj, n, ncols, G.hvec, G.hvec2, G, j, 0, true, 0)); }
                    k_select<<<1, 32, sizeof(double) * 3 * (m + 2), c->stream>>>(G, G.hvec, G.hvec2, j, ncols, eta * eta);
                    c->stats.kernel_launches++;
                    { ProfScope ps(c, 3, "gmres_wmvh (w-=V h update [+norm+Givens])", (8.0 * ncols + 16.0) * n);
                      KL_TRY(launch_wmvh(c, V, ldv, wj, n, ncols, G.hvec2, true, G, j, true, true, true)); }
                    bytes += (24.0 * ncols + 40.0) * n;
                } else if (coop) {
                    KL_TRY(launch_cgs2_coop(c, V, ldv, m + 1, wj, n, ncols, G, j));
                    bytes += (24.0 * ncols + 40.0) * n;
                } else if (ts_tma_ok(c, n, ldv, ncols, P.nx, P.ny)) {
                    // 3 passes over V: project ; update + project (fused, V tile staged once) ; update + norm
                    { ProfScope ps(c, 2, "gmres_vtw_tma (h1=V^T w, TMA-staged tall-skinny projection)", (8.0 * ncols + 8.0) * n);
                      KL_TRY(launch_ts_tma(c, false, V, ldv, m + 1, wj, n, ncols, nullptr, G.hvec, G, j, 1, true)); }
                    { ProfScope ps(c, 4, "gmres_wmvh_vtw_tma (w-=V h1 fused with h2=V^T w)", (8.0 * ncols + 16.0) * n);
                      KL_TRY(launch_ts_tma(c, true, V, ldv, m + 1, wj, n, ncols, G.hvec, G.hvec2, G, j, 2, true)); }
                    { ProfScope ps(c, 3, "gmres_wmvh (w-=V h update [+norm+Givens])", (8.0 * ncols + 16.0) * n);
                      KL_TRY(launch_wmvh(c, V, ldv, wj, n, ncols, G.hvec2, true, G, j, true, true)); }
                    bytes += (24.0 * ncols + 40.0) * n;
                } else {
                { ProfScope ps(c, 2, "gmres_vtw (h=V^T w tall-skinny projection)", (8.0 * ncols + 8.0) * n);
                  KL_TRY(launch_vtw(c, V, ldv, wj, n, ncols, G.hvec, G, j, 1, true)); }
                { ProfScope ps(c, 3, "gmres_wmvh (w-=V h update [+norm+Givens])", (8.0 * ncols + 16.0) * n);
                  KL_TRY(launch_wmvh(c, V, ldv, wj, n, ncols, G.hvec, false, G, j, false, true)); }
                { ProfScope ps(c, 2, "gmres_vtw (h=V^T w tall-skinny projection)", (8.0 * ncols + 8.0) * n);
                  KL_TRY(launch_vtw(c, V, ldv, wj, n, ncols, G.hvec, G, j, 2, true)); }
                { ProfScope ps(c, 3, "gmres_wmvh (w-=V h update [+norm+Givens])", (8.0 * ncols + 16.0) * n);
                  KL_TRY(launch_wmvh(c, V, ldv, wj, n, ncols, G.hvec, true, G, j, true, true)); }
                bytes += (32.0 * ncols + 48.0) * n;
                }
            }
            bytes += (24.0 + ((prec && !chain_step) ? 16.0 : 0.0)) * n;
            norm_idx = S_HVAL;
        }
        // V_{m+1} = w / h_val (:384).  omp: also on the converged step ; mf: not (:172-176)
        {
            PScale s;
            set_gate(s, c, true, m - 1, mf ? 0 : 1);
            s.in = w; s.out = V + (size_t)m * ldv; s.S = c->d_S; s.s_idx = S_HVAL;
            KL_TRY(launch_pointwise(c, s, n, NoPost{}));
        }
        KL_TRY(launch_backsolve(c, G));                                               // :394-398
        if (vec == 2) k_xpvy<2><<<upd_grid(n / 2), kTsThreads, sizeof(double) * m, c->stream>>>(V, ldv, dx, n, G);
        else k_xpvy<1><<<upd_grid(n), kTsThreads, sizeof(double) * m, c->stream>>>(V, ldv, dx, n, G);
        c->stats.kernel_launches += 1;
        return KL_OK;
    };
    const bool use_graph = c->opt_use_graph && !c->opt_profile && c->nranks == 1 && fused &&
                           (P.pc.kind == KL_PC_NONE || P.pc.kind == KL_PC_CBPR2 || P.pc.kind == KL_PC_CHEB);
    GraphKey gk;
    if (use_graph) {
        gk.add('G').add(nx).add(ny).add(m).add(mf).add(P.op.kind).add(P.op.eps_x).add(P.op.eps_y).add(P.w5).add(P.pc.kind)
            .add(P.pc.degree).add(P.params).add(c->opt_ortho).add(c->opt_reorth_eta_permille).add(c->opt_tma)
            .add(c->opt_chain).add(c->opt_stencil_rows).add(c->opt_stencil_tail).add(c->opt_stencil_stagger)
            .add(c->opt_pdl).add(c->opt_coop).add(c->opt_reverse).add(c->opt_persistent).add(c->ws).add(db).add(dx).add(V).add(G.H);
    }
    for (int st = 1; st <= max_restarts; ++st) {
        ++cycles;
        Ctx::GraphEntry *ge = use_graph ? graph_find(c, gk.s) : nullptr;
        if (use_graph && !ge && st >= 2) {
            // (the first cycle of a handle's first solve runs eagerly: it sets the function attributes and fills
            // the tensor-map cache)
            const double b0 = bytes;
            const long long l0 = c->stats.kernel_launches;
            KL_TRY(graph_begin(c));
            const int rc = enqueue_cycle();
            if (rc < 0) {
                Ctx::GraphEntry *dummy = nullptr;
                graph_end(c, std::string(), 0.0, 0, &dummy);
                graph_clear(c);
                return rc;
            }
            KL_TRY(graph_end(c, gk.s, bytes - b0, c->stats.kernel_launches - l0, &ge));
            bytes = b0;
            c->stats.kernel_launches = l0;
        }
        if (ge) {
            KL_CUDA(c, cudaGraphLaunch(ge->exec, c->stream));
            bytes += ge->bytes;
            c->stats.kernel_launches += ge->launches;
        } else {
            KL_TRY(enqueue_cycle());
        }
        KL_TRY(read_back(c));
        n_out = c->h_pinned_i[I_NOUT];
        bytes += (8.0 * n_out + 16.0) * n;
        const double h_val = c->h_pinned[S_HVAL], fe = c->h_pinned[S_RES];
        if (c->h_pinned_i[I_BREAKDOWN]) { status = KL_BREAKDOWN; restart_out = st; break; }
        if (h_val < tol || fe < tol) {                                               // :409-412
            restart_out = st;
            status = KL_OK;
            break;
        }
    }
    KL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    // mf variant: the converged step leaves V(:,n_out+1) = 0 (exit precedes :176; V = 0 at :128)
    if (mf && c->h_pinned_i[I_CONV_AT] >= 0)
        KL_CUDA(c, cudaMemsetAsync(V + (size_t)(c->h_pinned_i[I_CONV_AT] + 1) * ldv, 0, n * sizeof(double), c->stream));
    KL_TRY(stage_out(c, x, dx, n));
    KL_CUDA(c, cudaMemcpyAsync(final_err, G.fe, sizeof(double) * m, cudaMemcpyDeviceToHost, c->stream));
    KL_TRY(fetch_history(c));
    for (int i = 0; i <= m; ++i) v_err[i] = 0.0;
    c->stats.orth_frobenius = NAN;
    if (c->opt_verr && n_out >= 1) {
        // gmres_mgsr.f90:414-420 on the last cycle's basis, columns 0..n_out
        const int k = n_out + 1;
        std::vector<double> gr;
        KL_TRY(gram_lower(c, V, ldv, n, k, d_gram, gr));
        double fro = 0.0;
        for (int col = 0; col < k; ++col)
            for (int i = 0; i <= col; ++i) {
                double d = gr[(size_t)col * k + i] - (i == col ? 1.0 : 0.0);
                fro += (i == col ? 1.0 : 2.0) * d * d;
            }
        c->stats.orth_frobenius = sqrt(fro);
        for (int j = 0; j < n_out; ++j) {
            for (int i = 0; i <= j; ++i) {
                double d = gr[(size_t)(j + 1) * k + i];
                v_err[j + 1] = v_err[j + 1] + 2.0 * (d * d);
            }
            double dd = gr[(size_t)(j + 1) * k + (j + 1)] - 1.0;
            v_err[j + 1] = v_err[j + 1] + dd * dd;
            v_err[j + 1] = sqrt(v_err[j] * v_err[j] + v_err[j + 1]);
        }
    }
    KL_CUDA(c, cudaEventRecord(evB, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    KL_CUDA(c, cudaGetLastError());
    prof_resolve(c);
    float ms = 0, ms_tot = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    cudaEventElapsedTime(&ms_tot, evA, evB);
    c->stats.iterations = c->h_pinned_i[I_ITER];
    c->stats.cycles = cycles;
    c->stats.solve_ms = ms;
    c->stats.total_ms = ms_tot;
    // selective reorthogonalisation: the skipped second update passes moved no data (neither in the per-iteration
    // total nor in the per-kernel profile, where every launch was charged when it was enqueued)
    const double skipped_bytes = (8.0 * c->h_pinned_i[I_NSKIPCOLS] + 16.0 * c->h_pinned_i[I_NSKIP]) * (double)n;
    bytes -= skipped_bytes;
    if (c->opt_profile && c->prof_launches[3] > 0) {
        c->prof_bytes[3] -= skipped_bytes;
        c->prof_launches[3] -= c->h_pinned_i[I_NSKIP];      // launches that returned at once are not counted
        if (c->prof_launches[3] < 1) c->prof_launches[3] = 1;
    }
    c->stats.algorithmic_bytes = bytes;
    c->stats.reorth_skipped = c->h_pinned_i[I_NSKIP];
    *n_out_p = n_out;
    *restart_out_p = restart_out;
    return status;
}

}  // namespace kl

using namespace kl;

extern "C" {

int kl_gmres_mgsr_omp(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                      int m, double tol, double *final_err, double *v_err, int *n_out, int *restart_out,
                      const kl_precond_t *M, const double *params, int nparams) {
    return gmres_mgsr_solve(h, A, b, x, nx, ny, m, tol, final_err, v_err, n_out, restart_out, M, params,
                            nparams, 0);
}
int kl_gmres_mgsr_mf(kl_handle_t h, const kl_operator_t *A, const double *b, double *x, int nx, int ny,
                     int m, double tol, double *final_err, double *v_err, int *n_out, int *restart_out,
                     const kl_precond_t *M, const double *params, int nparams) {
    return gmres_mgsr_solve(h, A, b, x, nx, ny, m, tol, final_err, v_err, n_out, restart_out, M, params,
                            nparams, 1);
}

}  // extern "C"
