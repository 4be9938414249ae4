// kl_csr.cu -- the sparse-matrix operator KL_OP_CSR: y = A x, Jacobi-scaled Chebyshev steps on it, and the check of
// its index arrays.
//
// Evaluation order (krylov_b200.h kl_csr_t; tests/csr_twin.c reproduces it bit for bit): one matrix-wide width W, the
// smallest power of two >= ceil(nnz / n) clamped to [1, 32].  Row i is served by W consecutive lanes of a warp; lane l
// sums k = row_ptr[i] + l, + W, ... in storage order with fma, and an xor butterfly over the W lanes combines the
// partial sums.  A row is served by one W-lane group whatever its length (no merge-path balancing): a row of 10^4
// entries costs its group 10^4 / W steps while the rest of the matrix streams past it.
//
// Traffic per application: val and col_ind (12 nnz B) and row_ptr (8(n+1) B) are read once, x is gathered (8n B if
// every value is fetched from HBM once) and y written (8n B).  All loads are plain read-only loads: PTX cache-policy
// hints (val and col_ind evict-first past L1, x evict-last in L2) measured 1-3 % slower on a B200 at every size of
// scripts/csr_bench.py (profiles/r09_csr.json), because the kernel is bound by the latency of its dependent loads
// (row_ptr, then col_ind and val, then x), not by what L2 keeps.
//
// Safety: the index arrays are outside input.  Whatever they hold, no load leaves [0, nnz) or [0, n): a row range is
// clamped to [0, nnz] and a column is compared unsigned against n, an out-of-range entry contributing nothing.
// k_csr_check finds such input before a solve (csr_validate) and the call returns KL_ERR_INVALID.
#include "kl_ops.cuh"

namespace kl {

static constexpr int kCsrBlock = 256;
// Rows per W-lane group.  One row per group leaves a lane with a single chain of three dependent loads (row_ptr, then
// col_ind and val, then x) and the kernel latency-bound at 23 % of the HBM rate on CSR Poisson; R rows whose loads are
// issued together put R chains in flight per lane.
static constexpr int kCsrRows = 4;

// The rows of a lane: warp w serves rows [w R G, (w+1) R G), G = 32 / W groups of W lanes; group g takes rows
// w R G + r G + g, r < R, so that the groups of a warp read neighbouring rows at each r.
template <int W>
__device__ __forceinline__ long long csr_row0(int &lane) {
    constexpr int G = 32 / W;
    const long long warp = ((long long)blockIdx.x * kCsrBlock + threadIdx.x) / 32;
    const int l32 = threadIdx.x & 31;
    lane = l32 % W;
    return warp * kCsrRows * G + l32 / W;
}

// The W-lane scan of the rows row0 + r G, r < R, shared by the kernels.  DOT: s[r] = sum val[k] x[col[k]] in the
// documented order.  DIAG: dg[r] = the sum of the row's diagonal entries (each lane adds its own in storage order, then
// the butterfly), hs[r] != 0 iff the row stores one.  Every lane of the group returns the same values.  All lanes of
// the warp must call it (shuffles).
template <int W, bool DOT, bool DIAG>
__device__ __forceinline__ void rows_scan(const kl_csr_t m, const int n, const long long row0, const int lane,
                                          const double *__restrict__ x, double (&s)[kCsrRows],
                                          double (&dg)[kCsrRows], int (&hs)[kCsrRows]) {
    constexpr int R = kCsrRows, G = 32 / W;
    long long k[R], hi[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long i = row0 + (long long)r * G;
        long long lo = 0, h = 0;
        if (i < n) {
            lo = __ldg(reinterpret_cast<const long long *>(m.row_ptr) + i);
            h = __ldg(reinterpret_cast<const long long *>(m.row_ptr) + i + 1);
        }
        lo = lo < 0 ? 0 : (lo > m.nnz ? m.nnz : lo);
        k[r] = lo + lane;
        hi[r] = h > m.nnz ? m.nnz : h;
        s[r] = 0.0;
        dg[r] = 0.0;
        hs[r] = 0;
    }
    // step j takes entry row_ptr[i] + lane + j W of every row that has one: the R rows' loads are in flight together,
    // and each row's sum still runs in storage order
    for (;;) {
        int c[R];
        double v[R], xv[R];
        bool ok[R], any = false;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            ok[r] = k[r] < hi[r];
            any |= ok[r];
            c[r] = ok[r] ? __ldg(m.col_ind + k[r]) : -1;
            v[r] = ok[r] ? __ldg(m.val + k[r]) : 0.0;
        }
        if (!any) break;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            ok[r] = ok[r] && (unsigned)c[r] < (unsigned)n;
            if (DOT) xv[r] = ok[r] ? __ldg(x + c[r]) : 0.0;
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (ok[r]) {
                if (DOT) s[r] = fma(v[r], xv[r], s[r]);
                if (DIAG && c[r] == row0 + (long long)r * G) { dg[r] += v[r]; hs[r] = 1; }
            }
            k[r] += W;
        }
    }
#pragma unroll
    for (int off = W / 2; off >= 1; off /= 2) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (DOT) s[r] = s[r] + __shfl_xor_sync(0xffffffffu, s[r], off);
            if (DIAG) {
                dg[r] = dg[r] + __shfl_xor_sync(0xffffffffu, dg[r], off);
                hs[r] |= __shfl_xor_sync(0xffffffffu, hs[r], off);
            }
        }
    }
}

template <int W>
static unsigned csr_blocks(int n) {
    constexpr int rows_per_block = kCsrBlock / W * kCsrRows;
    return (unsigned)(((size_t)n + rows_per_block - 1) / rows_per_block);
}

// y = A x.  12 nnz + 8(n+1) + 8n + 8n B.
template <int W>
__global__ void __launch_bounds__(kCsrBlock, 4)
k_csr_spmv(const kl_csr_t m, const int n, const double *__restrict__ x, double *__restrict__ y,
           const int *__restrict__ flags) {
    if (flags && flags[I_CONV_AT] >= 0) return;
    int lane;
    const long long row0 = csr_row0<W>(lane);
    double s[kCsrRows], dg[kCsrRows];
    int hs[kCsrRows];
    rows_scan<W, true, false>(m, n, row0, lane, x, s, dg, hs);
    if (lane != 0) return;
#pragma unroll
    for (int r = 0; r < kCsrRows; ++r) {
        const long long i = row0 + (long long)r * (32 / W);
        if (i < n) y[i] = s[r];
    }
}

// Jacobi-scaled Chebyshev on KL_OP_CSR, one pass per step: the per-point arithmetic of k_jacobi_cheb_step (kl_ops.cu)
// with A z and a_ii from the row scan and dinv = RN(1/a_ii) recomputed in every pass.
// kind 2: z = r*dinv ; kind 1: the start, d = z = (r*dinv)/theta ; kind 0: one step,
// d = fma(c1, d, c2*((r - A zin)*dinv)), z = zin + d.
template <int W>
__global__ void __launch_bounds__(kCsrBlock, 4)
k_csr_jacobi_cheb_step(const kl_csr_t m, const int n, const double *__restrict__ r, const double *__restrict__ zin,
                       double *__restrict__ d, double *__restrict__ z, const double theta, const double c1,
                       const double c2, const int kind, const int *__restrict__ flags) {
    if (flags && flags[I_CONV_AT] >= 0) return;
    int lane;
    const long long row0 = csr_row0<W>(lane);
    double az[kCsrRows], dg[kCsrRows];
    int hs[kCsrRows];
    if (kind == 0) rows_scan<W, true, true>(m, n, row0, lane, zin, az, dg, hs);
    else rows_scan<W, false, true>(m, n, row0, lane, nullptr, az, dg, hs);
    if (lane != 0) return;
#pragma unroll
    for (int q = 0; q < kCsrRows; ++q) {
        const long long i = row0 + (long long)q * (32 / W);
        if (i >= n) continue;
        const double dinv = __drcp_rn(dg[q]), rc = __ldg(r + i);
        if (kind == 2) {
            z[i] = rc * dinv;
        } else if (kind == 1) {
            const double d0 = (rc * dinv) / theta;
            d[i] = d0;
            z[i] = d0;
        } else {
            const double dn = fma(c1, d[i], c2 * ((rc - az[q]) * dinv));
            d[i] = dn;
            z[i] = __ldg(zin + i) + dn;
        }
    }
}

// bad |= 1: row_ptr[0] != 0, row_ptr decreasing, row_ptr[n] != nnz or a column outside [0, n) ;
// bad |= 2 (jacobi): a row without a diagonal entry or with a zero one.
// Reads row_ptr[0..n], col_ind[0..nnz) and (jacobi) the diagonal values only.
template <int W>
__global__ void __launch_bounds__(kCsrBlock)
k_csr_check(const kl_csr_t m, const int n, const int jacobi, int *__restrict__ bad) {
    const size_t t = (size_t)blockIdx.x * kCsrBlock + threadIdx.x;
    const int i = (int)(t / W), lane = (int)(t % W);
    int err = 0;
    double dg = 0.0;
    int hs = 0;
    if (i < n) {
        const long long lo0 = m.row_ptr[i], hi0 = m.row_ptr[i + 1];
        if (lane == 0 && ((i == 0 && lo0 != 0) || lo0 > hi0 || (i == n - 1 && hi0 != m.nnz))) err = 1;
        const long long lo = lo0 < 0 ? 0 : (lo0 > m.nnz ? m.nnz : lo0), hi = hi0 > m.nnz ? m.nnz : hi0;
        for (long long k = lo + lane; k < hi; k += W) {
            const int col = m.col_ind[k];
            if ((unsigned)col >= (unsigned)n) err = 1;
            else if (jacobi && col == i) { dg += m.val[k]; hs = 1; }
        }
    }
#pragma unroll
    for (int off = W / 2; off >= 1; off /= 2) {
        dg = dg + __shfl_xor_sync(0xffffffffu, dg, off);
        hs |= __shfl_xor_sync(0xffffffffu, hs, off);
    }
    if (jacobi && lane == 0 && i < n && (!hs || dg == 0.0)) err |= 2;
    if (err) atomicOr(bad, err);
}

template <int W>
static unsigned csr_check_blocks(int n) {
    return (unsigned)(((size_t)n * W + kCsrBlock - 1) / kCsrBlock);
}

int csr_width(int n, long long nnz) {
    const long long per = n > 0 ? (nnz + n - 1) / n : 0;
    int w = 1;
    while (w < 32 && w < per) w *= 2;
    return w;
}

#define KL_CSR_SWITCH(W_, CALL)                                            \
    switch (W_) {                                                          \
        case 1: { constexpr int W = 1; CALL; } break;                      \
        case 2: { constexpr int W = 2; CALL; } break;                      \
        case 4: { constexpr int W = 4; CALL; } break;                      \
        case 8: { constexpr int W = 8; CALL; } break;                      \
        case 16: { constexpr int W = 16; CALL; } break;                    \
        default: { constexpr int W = 32; CALL; } break;                    \
    }

int launch_csr_spmv(Ctx *c, const kl_csr_t *m, int n, const double *x, double *y, bool gated) {
    const int *flags = gated ? c->d_I : nullptr;
    KL_CSR_SWITCH(csr_width(n, m->nnz),
                  (k_csr_spmv<W><<<csr_blocks<W>(n), kCsrBlock, 0, c->stream>>>(*m, n, x, y, flags)));
    c->stats.kernel_launches++;
    return KL_OK;
}

int launch_csr_jacobi_cheb_step(Ctx *c, const kl_csr_t *m, int n, const double *r, const double *zin, double *d,
                                double *z, double theta, double c1, double c2, int kind, bool gated) {
    const int *flags = gated ? c->d_I : nullptr;
    KL_CSR_SWITCH(csr_width(n, m->nnz),
                  (k_csr_jacobi_cheb_step<W><<<csr_blocks<W>(n), kCsrBlock, 0, c->stream>>>(
                      *m, n, r, zin, d, z, theta, c1, c2, kind, flags)));
    c->stats.kernel_launches++;
    return KL_OK;
}

int csr_validate(Ctx *c, const kl_csr_t *m, int n, bool jacobi) {
    int *bad = c->d_I + I_CSR_BAD;
    KL_CUDA(c, cudaMemsetAsync(bad, 0, sizeof(int), c->stream));
    KL_CSR_SWITCH(csr_width(n, m->nnz),
                  (k_csr_check<W><<<csr_check_blocks<W>(n), kCsrBlock, 0, c->stream>>>(*m, n, jacobi ? 1 : 0, bad)));
    c->stats.kernel_launches++;
    KL_CUDA(c, cudaGetLastError());
    KL_CUDA(c, cudaMemcpyAsync(c->h_pinned_i + I_CSR_BAD, bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    KL_CUDA(c, cudaStreamSynchronize(c->stream));
    const int e = c->h_pinned_i[I_CSR_BAD];
    if (e & 1)
        return c->fail(KL_ERR_INVALID, "KL_OP_CSR: malformed matrix (row_ptr[0] != 0, row_ptr decreasing, "
                                       "row_ptr[n] != nnz, or a column outside [0, n))");
    if (e & 2) return c->fail(KL_ERR_INVALID, "KL_PC_JACOBI_CHEB on KL_OP_CSR: a diagonal entry is missing or zero");
    return KL_OK;
}

#undef KL_CSR_SWITCH

}  // namespace kl
