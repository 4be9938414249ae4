// kl_internal.cuh -- shared internals of libkrylov_b200 (sm_100a only).
//
// Design notes (see DESIGN.md):
//  * every kernel is FP64 and HBM-bound; no tensor cores on this path.
//  * compiled with -fmad=false: every fused multiply-add is written as an
//    explicit fma() so that point-wise results are bit-identical to the CPU
//    oracle's (which is compiled with -ffp-contract=off and the same fma()s).
//  * reductions are deterministic: per-block partial sums in a fixed order,
//    summed by the last block to finish (threadfence + counter) in a fixed
//    order.  The same launch configuration gives the same bits every run.
//  * solver scalars (alpha, beta, Givens data, convergence flag, iteration
//    counters, residual history) live in device memory; "post" functors run in
//    the last block of the reducing kernel (single GPU) or in a 1-thread kernel
//    after the NCCL all-reduce (multi GPU).  The host never sits between two
//    kernels of an iteration.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/krylov_b200.h"

namespace kl {

// ------------------------------------------------------------------------
// limits
// ------------------------------------------------------------------------
constexpr int kMaxRed = 8;          // reductions per point-wise / stencil kernel
constexpr int kMaxBlocks = 16384;    // upper bound on reducing-kernel grid size (partials leading dimension)
constexpr int kMaxCols = 512;       // max restart length m+1 supported by the tall-skinny kernels
constexpr int kNumSM = 148;
constexpr int kMaxDevices = 16;      // per-device launch state (function attributes, occupancy)

// device scalar block layout (doubles)
enum SIdx {
    S_ALPHA = 0, S_BETA, S_OMEGA, S_RR, S_PAP, S_RES, S_TOL, S_BETA0, S_HVAL, S_NORM, S_TMP0,
    S_TMP1, S_TMP2, S_TMP3, S_CD, S_CALPHA, S_RHO, S_RHOPREV, S_C1, S_C2, S_THETA, S_SCALE,
    S_ALPHA_PREV, S_BETA_PREV,     // CG pair mode: alpha and beta of the previous iteration (cg_onepass_scalars)
    S_RED = 32,            // kMaxRed all-reduced sums land here (S_RED .. S_RED+7)
    S_LAN = 64,            // lanczos alphas/betas etc.
    S_COUNT = 1024
};
// device int block layout
enum IIdx {
    I_CONV_AT = 0,   // -1: running ; >=0: step/iteration index at which convergence was detected
    I_ITER,          // iterations completed (CG/BiCGSTAB) / total inner iterations (GMRES)
    I_NOUT,          // GMRES n_out of the current cycle
    I_HIST,          // number of history entries written
    I_BREAKDOWN,
    I_STEP,
    I_SKIP3,         // selective reorthogonalisation: 1 = the second update pass of this step is skipped
    I_NSKIP,         // number of skipped second passes ; I_NSKIPCOLS = sum of their column counts
    I_NSKIPCOLS,
    I_COUNT = 64
};

}  // namespace kl
#include "kl_posts.cuh"
namespace kl {

// NVLink peer-memory communication buffer (one per rank, mapped into every process through CUDA IPC); layout in
// doubles.  Used by the stand-alone collectives in kl_core.cu and by the all-reduce that the LAST BLOCK of a
// reducing kernel performs inline (peer_allreduce_block below).
constexpr int kArMax = 128;                 // doubles per all-reduce
constexpr int kHaloNxCap = 65536;           // widest halo message (doubles) supported by the peer path
constexpr size_t kCbArInbox = 0;                                        // [2][16][kArMax] doubles
constexpr size_t kCbArFlags = kCbArInbox + 2 * 16 * kArMax;             // [2][16] u64
constexpr size_t kCbHaloFlags = kCbArFlags + 2 * 16;                    // [2][4 slots][2 dirs] u64
constexpr size_t kCbHalo = kCbHaloFlags + 2 * 4 * 2;                    // [2][4][2][kHaloNxCap] doubles
// halo lines PUSHED BY THE PRODUCING KERNEL (edge CTAs of a stencil kernel store the first / last line of an
// output vector straight into the neighbours' slots; the all-reduce that ends the same kernel is the barrier that
// makes them visible before any consumer starts, so there is no halo kernel and no halo flag on that path)
constexpr int kPushSlots = 4;
constexpr size_t kCbPush = kCbHalo + (size_t)2 * 4 * 2 * kHaloNxCap;   // [2 parity][kPushSlots][2 dirs][kHaloNxCap]
constexpr size_t kCbDoubles = kCbPush + (size_t)2 * kPushSlots * 2 * kHaloNxCap;
constexpr long long kSpinLimit = 1ll << 27;   // ~seconds: a lost peer flags a breakdown instead of hanging
struct PeerCtl {             // lives in device memory (RedCtl carries a pointer to it)
    double *p[16];           // every rank's communication buffer
    int rank, nranks;
    // sequence number of the last EXECUTED all-reduce.  Device-resident on purpose: kernels that are gated off
    // after convergence never take part in a collective, so a host-side counter would run ahead of the
    // collectives that really happened and two executed all-reduces could share a parity slot with no
    // cross-rank barrier between them.  Every rank executes the same collectives, so the counters agree.
    unsigned long long ar_seq;
};
__host__ __device__ inline size_t push_slot_off(int parity, int slot, int dir) {
    return kCbPush + (((size_t)parity * kPushSlots + slot) * 2 + dir) * kHaloNxCap;
}

struct RedCtl {
    double *partials;        // [grid * ld]
    unsigned int *counter;   // zero between kernels
    double *red;             // local sums destination
    PeerCtl *peer;           // != nullptr: the last block all-reduces `red` over NVLink before the post functor
    int *I;                  // int block (breakdown flag for a lost peer)
};

// ------------------------------------------------------------------------
// host context
// ------------------------------------------------------------------------
}  // namespace kl
struct kl_context_s;
namespace kl {
using Ctx = ::kl_context_s;
int comm_allreduce(Ctx *c, double *d_buf, int count);
// exchanges the boundary lines of nvec slab vectors; lo_out/hi_out receive the halo line pointers
// (nullptr at the global boundary)
int comm_halo_exchange(Ctx *c, const double *const *send_lo_rows, const double *const *send_hi_rows,
                       const double **lo_out, const double **hi_out, int nvec, int nx);
// "producer pushes" halo scheme (kl_core.cu)
bool comm_push_ok(const Ctx *c, int count);
void comm_push_recv(const Ctx *c, int parity, int slot, const double **lo, const double **hi);
void comm_push_send(const Ctx *c, int parity, int slot, double **first_dst, double **last_dst);
int comm_push_lines(Ctx *c, int nvec, const double *const *first, const double *const *last, const int *slots,
                    int parity, int count);

}  // namespace kl

struct kl_context_s {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    int pointer_mode = KL_POINTER_HOST;
    std::string err;
    // options
    int opt_ortho = KL_ORTHO_CGS2;
    int opt_max_restarts = 1000;
    int opt_verr = 1;
    int opt_check_every = 32;
    int opt_use_graph = 1;
    int opt_hh_mode = KL_HH_BLOCKED;
    int opt_fuse = 1;
    int opt_profile = 0;
    int opt_tma = 1;
    int pdl_scope = 0;           // > 0: every PDL-capable launch uses programmatic dependent launch (PdlScope)
    long long opt_chain_step_min = 1 << 20;   // one-pass GMRES step (ChGmresStep) from this many local unknowns on (env KL_CHAIN_STEP_MIN)
    int opt_chain_rows_min = 0;  // > 0: lower bound of the chain kernels' lines per CTA on small grids (env KL_CHAIN_ROWS_MIN)
    int opt_ts_blocks = 0;       // > 0: cap on the CTAs of the tall-skinny passes (tuning; env KL_TS_BLOCKS)
    int opt_chain = 1;          // temporally blocked (chained) stencil kernels, kl_chain_tma.cuh
    int opt_reorth_eta_permille = 300;   // KL_ORTHO_CGS2_SELECTIVE: reorthogonalise iff ||w'|| < eta ||w||.  0.3 from the sweep in
                                         // profiles/r02_eta_sweep.json (identical iteration counts for every eta <= 0.707 on
                                         // 1024^2..4096^2, ||I - V^T V|| <= 2e-12); 707 = 1/sqrt 2 is Kahan-Parlett's bound
    int opt_stencil_rows = 0;   // 0: heuristic
    int opt_persistent = 0;      // persistent CTAs in the TMA stencil kernels (KL_OPT_PERSISTENT): measured 4-8 % slower
                                 // than one CTA per tile (static tile assignment balances worse than the hardware's
                                 // dynamic CTA scheduling, profiles/r02_cta_timeline_persistent.txt): off by default
    int opt_persist_occ = 0;     // CTAs per SM of the persistent grid (0 = full occupancy)
    int opt_coop = 0;            // cooperative one-kernel CGS2 step on small grids (KL_OPT_COOP).  Measured at 300^2 against
                                 // three graph-replayed launches: 4 % slower with cooperative_groups grid barriers, 1.6 %
                                 // faster (43.5 vs 44.2 us per step) with the arrival-counter + flag barriers it has now:
                                 // the step is bound by what happens INSIDE a pass, not by launches.  Off.
    int opt_reverse = 0;         // K2-type kernels march against their predecessor's direction (KL_OPT_REVERSE): no
                                 // measurable L2 reuse on B200 (264.0 vs 265.0 us at 8 GPUs): off by default
    int opt_stencil_stagger = 0; // staggered tile heights (KL_OPT_STENCIL_STAGGER): measured neutral, off by default
    int opt_stencil_tail = -1;  // lines per CTA in the tapered tail (-1 auto, 0 off), KL_OPT_STENCIL_TAIL
    int opt_pdl = 1;            // programmatic dependent launch between the fused CG kernels (KL_OPT_PDL)
    int opt_cg_onepass = -1;    // plain CG in chain passes (KL_OPT_CG_ONEPASS): -1 auto, 0 off, 1 one pass per iteration, 2 pairs
    int opt_x0 = 0;             // x is the initial guess on entry (KL_OPT_X0); no environment variable: it turns an output
                                // into an input
    // comm
    int rank = 0, nranks = 1;
    void *nccl_comm = nullptr;
    // NVLink peer-memory collectives (one-shot all-reduce and halo push over IPC-mapped buffers)
    int opt_peer = 1;
    bool peer_ok = false;
    bool peer_mapped = false;            // every rank mapped every peer buffer (peer_setup agreed)
    int opt_push_halo = 1;               // producing kernels push their boundary lines (KL_OPT_PUSH_HALO)
    double *cb_local = nullptr;          // this rank's communication buffer
    double *cb_peer[16] = {};            // every rank's buffer mapped into this process (cb_peer[rank] = cb_local)
    unsigned long long halo_seq = 0;
    struct kl::PeerCtl *d_peerctl = nullptr;   // device copy of the peer pointers (inline all-reduce)
    int opt_inline_ar = 1;                     // all-reduce inside the reducing kernel's last block
    // device blocks
    double *d_S = nullptr;
    int *d_I = nullptr;
    double *d_partials = nullptr;
    unsigned int *d_counter = nullptr;
    double *d_hist = nullptr;
    int hist_cap = 0;
    double *h_pinned = nullptr;   // pinned mirror for scalar read-back
    int *h_pinned_i = nullptr;
    // workspace arena (grown on demand, reused across calls)
    char *ws = nullptr;
    size_t ws_bytes = 0, ws_used = 0;
    // halo buffers (multi GPU): up to 4 vectors x 2 directions
    double *d_halo = nullptr;
    size_t halo_doubles = 0;
    // CUDA-graph replay of iteration batches / restart cycles (KL_OPT_USE_GRAPH): executable graphs cached by a
    // key that holds everything baked into the captured launches (problem, options, buffer addresses)
    struct GraphEntry { std::string key; cudaGraphExec_t exec; double bytes; long long launches; };
    std::vector<GraphEntry> graphs;
    cudaStream_t cap_stream = nullptr;     // capture happens here (the user stream may be the legacy stream)
    cudaStream_t saved_stream = nullptr;
    bool capturing = false;
    // stats
    kl_stats_t stats{};
    std::vector<double> history;
    int history_len = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // iteration loop
    cudaEvent_t ev2 = nullptr, ev3 = nullptr;   // whole call (incl. host<->device copies)
    // TMA descriptor cache (opaque 128-byte CUtensorMap blobs keyed by base pointer and extents)
    struct TmapEntry { const void *base; int nx, ny; long long k1 = 0, k2 = 0; alignas(64) unsigned char blob[128]; };
    std::vector<TmapEntry> tmaps;
    void *encode_fn = nullptr;
    // profiling (KL_OPT_PROFILE): event pairs per kernel class, resolved after the solve
    struct ProfRec { int cls; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> prof_pool;
    const char *prof_name[KL_PROFILE_CLASSES] = {};
    double prof_ms[KL_PROFILE_CLASSES] = {};
    long long prof_launches[KL_PROFILE_CLASSES] = {};
    double prof_bytes[KL_PROFILE_CLASSES] = {};

    int fail(int code, const char *what, cudaError_t e = cudaSuccess) {
        char buf[512];
        snprintf(buf, sizeof buf, "%s%s%s", what, e != cudaSuccess ? ": " : "",
                 e != cudaSuccess ? cudaGetErrorString(e) : "");
        err = buf;
        return code;
    }
};

namespace kl {

#define KL_CUDA(c, call)                                                     \
    do {                                                                     \
        cudaError_t e__ = (call);                                            \
        if (e__ != cudaSuccess) return (c)->fail(KL_ERR_CUDA, #call, e__);   \
    } while (0)
#define KL_TRY(call)                 \
    do {                             \
        int r__ = (call);            \
        if (r__ < 0) return r__;     \
    } while (0)

// profiling helpers (kl_core.cu)
void prof_reset(Ctx *c);
void prof_begin(Ctx *c, int cls, const char *name, double bytes);
void prof_end(Ctx *c);
void prof_resolve(Ctx *c);
struct ProfScope {
    Ctx *c;
    ProfScope(Ctx *c_, int cls, const char *name, double bytes) : c(c_) { if (c->opt_profile) prof_begin(c, cls, name, bytes); }
    ~ProfScope() { if (c->opt_profile) prof_end(c); }
};

// CUDA-graph helpers (kl_core.cu).  graph_find: cached executable graph or nullptr.  graph_begin redirects
// c->stream to the capture stream; graph_end instantiates, caches under `key` and restores c->stream.
Ctx::GraphEntry *graph_find(Ctx *c, const std::string &key);
int graph_begin(Ctx *c);
int graph_end(Ctx *c, const std::string &key, double bytes, long long launches, Ctx::GraphEntry **out);
void graph_clear(Ctx *c);
struct GraphKey {     // append-only byte string
    std::string s;
    template <class T> GraphKey &add(const T &v) { s.append(reinterpret_cast<const char *>(&v), sizeof(T)); return *this; }
};

// workspace arena
int ws_reserve(Ctx *c, size_t bytes);
inline void ws_reset(Ctx *c) { c->ws_used = 0; }
template <class T>
inline T *ws_take(Ctx *c, size_t count) {
    size_t off = (c->ws_used + 255) & ~size_t(255);
    c->ws_used = off + count * sizeof(T);
    return reinterpret_cast<T *>(c->ws + off);
}
inline size_t ws_need(size_t count, size_t elt = 8) { return ((count * elt) + 255 + 256) & ~size_t(255); }

// ------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// streaming loads / stores: data touched once per kernel -> do not pollute L1
__device__ __forceinline__ double2 ldg2(const double *p) {
    return __ldg(reinterpret_cast<const double2 *>(p));
}
__device__ __forceinline__ void stg2(double *p, double a, double b) {
    *reinterpret_cast<double2 *>(p) = make_double2(a, b);
}

// Correctly rounded x/d for a divisor that is constant over the kernel.
// The hardware sequence (MUFU.RCP64H + Newton steps + range check per element)
// makes division-carrying stencil kernels instruction-bound; with the reciprocal
// hoisted, Markstein's correction  q <- q + (x - q d) * rd  applied twice gives
// the IEEE-754 quotient in 5 FMA-class instructions (rd = RN(1/d); exact when no
// underflow/overflow occurs and the significand of d is not all ones -- those
// cases fall back to the hardware division).  Bit-compatibility with the
// reference's r(i)/d is verified in tests/test_gpu_parity.py.
static __device__ __noinline__ double slow_div(double x, double d) { return x / d; }
struct FastDiv {
    double d, rd;
    int ok;
    __host__ __device__ __forceinline__ void set(double dd) {
        d = dd;
        rd = 1.0 / dd;
        unsigned long long bits;
#ifdef __CUDA_ARCH__
        bits = (unsigned long long)__double_as_longlong(dd);
#else
        memcpy(&bits, &dd, sizeof bits);
#endif
        const unsigned long long man = bits & 0x000fffffffffffffULL;
        const int ex = (int)((bits >> 52) & 0x7ff);
        ok = (man != 0x000fffffffffffffULL) && ex > 200 && ex < 1800;
    }
    // two quotients with ONE warp-wide test for the rare operands (zero, tiny, huge, NaN): the common path is
    // straight-line code instead of a divergence scaffold (BSSY / BRA / BSYNC) per division.  All 32 lanes of the
    // warp must call it together.  The range test 2^-700 <= |x| < 2^700 runs on the exponent field in the integer
    // pipe (one shift-add and one unsigned compare per operand; `ok` is folded into the bounds by set()) instead
    // of two DSETP per operand on the half-rate FP64 pipe.
    __device__ __forceinline__ void div2(double x0, double x1, double &o0, double &o1) const {
        const double a0 = x0 * rd, a1 = x1 * rd;
        double r0 = fma(-a0, d, x0), r1 = fma(-a1, d, x1);
        double q0 = fma(r0, rd, a0), q1 = fma(r1, rd, a1);
        r0 = fma(-q0, d, x0);
        r1 = fma(-q1, d, x1);
        q0 = fma(r0, rd, q0);
        q1 = fma(r1, rd, q1);
        const unsigned lo2 = ok ? 2u * 0x14300000u : 0xffffffffu, span = ok ? 2u * (0x6bb00000u - 0x14300000u) : 0u;
        const bool in0 = (((unsigned)__double2hiint(x0) << 1) - lo2) < span;
        const bool in1 = (((unsigned)__double2hiint(x1) << 1) - lo2) < span;
        if (__any_sync(0xffffffffu, !(in0 && in1))) {
            if (!in0) q0 = (x0 == 0.0 && ok) ? a0 : slow_div(x0, d);
            if (!in1) q1 = (x1 == 0.0 && ok) ? a1 : slow_div(x1, d);
        }
        o0 = q0;
        o1 = q1;
    }
    __device__ __forceinline__ double div(double x) const {
        const double q0 = x * rd;
        double r = fma(-q0, d, x);
        double q = fma(r, rd, q0);
        r = fma(-q, d, x);
        q = fma(r, rd, q);
        const double ax = fabs(x);
        if (!(ok && ax >= 0x1p-700 && ax <= 0x1p700)) q = (x == 0.0 && ok) ? q0 : slow_div(x, d);
        return q;
    }
};

// Block-level reduction of K values, deterministic; result valid in thread 0.
template <int K, int NT>
__device__ __forceinline__ void block_sum(double (&v)[K], double *smem /* K * NT/32 */) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int NW = NT / 32;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double s = warp_sum(v[k]);
        if (lane == 0) smem[k * NW + wid] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            double s = 0.0;
            for (int w = 0; w < NW; ++w) s += smem[k * NW + w];
            v[k] = s;
        }
    }
}

// Grid-level deterministic reduction.  Every block calls this with its K block
// sums valid in thread 0.  Returns true in ALL threads of the last block to
// arrive, after red[0..K) holds the grid sums.  The last block sums the partials
// with all of its NT threads (thread t takes blocks t, t+NT, ... in increasing
// order, eight independent loads in flight), then combines the NT values in the
// fixed order of block_sum: same launch configuration => same bits.  `nblocks`
// is the linear grid size, `bid` the linear id, smem = K * NT/32 doubles.
template <int K, int NT>
__device__ __forceinline__ bool grid_sum(const double (&v)[K], const RedCtl &rc, unsigned nblocks,
                                         unsigned bid, int *s_flag, double *smem) {
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) rc.partials[(size_t)k * kMaxBlocks + bid] = v[k];
        __threadfence();
        unsigned prev = atomicAdd(rc.counter, 1u);
        *s_flag = (prev == nblocks - 1);
    }
    __syncthreads();
    if (!*s_flag) return false;
    __threadfence();
    double s[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const double *p = rc.partials + (size_t)k * kMaxBlocks;
        double a = 0.0;
        unsigned b = threadIdx.x;
        for (; b < nblocks; b += 8 * NT) {       // eight independent L2 loads in flight per thread; the ragged last
            double t[8];                        // round is predicated (adding +0.0 is exact), not a serial loop of
#pragma unroll                                  // dependent L2 round trips (~0.7 us each under load)
            for (int q = 0; q < 8; ++q) t[q] = (b + q * NT < nblocks) ? __ldcg(p + b + q * NT) : 0.0;
#pragma unroll
            for (int q = 0; q < 8; ++q) a += t[q];
        }
        s[k] = a;
    }
    block_sum<K, NT>(s, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) rc.red[k] = s[k];
        *rc.counter = 0u;
        __threadfence();
    }
    __syncthreads();
    return true;
}

__device__ __forceinline__ void st_release_sys(unsigned long long *addr, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *addr) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(addr) : "memory");
    return v;
}

// One-shot all-reduce of rc.red[0..K) over NVLink peer memory, executed by ALL threads of the last block of a
// reducing kernel (compute + collective in one kernel: no all-reduce launch, no post-functor launch).  Every
// rank pushes its sums into every rank's inbox with posted stores, raises a release flag carrying the sequence
// number, waits for the P flags and adds the inbox in rank order -- identical bits on every rank.  Same
// protocol, buffers and sequence counter as k_peer_allreduce (kl_core.cu), so both can be mixed in a stream.
// (__noinline__: inlined, its spin loops raised the register count of the point-wise kernels from 80 to 106,
// i.e. from 3 to 2 resident blocks per SM, and cost 40 % of their bandwidth on ONE GPU.)
template <int K>
__device__ __noinline__ void peer_allreduce_block(const RedCtl &rc) {
    PeerCtl &pc = *rc.peer;
    const unsigned long long seq = pc.ar_seq + 1ull;     // only this block touches it (kernels are stream-ordered)
    const int P = pc.nranks, rank = pc.rank, par = (int)(seq & 1ull);
    for (int t = threadIdx.x; t < K * P; t += blockDim.x) {
        const int q = t / K, i = t - q * K;
        pc.p[q][kCbArInbox + ((size_t)par * 16 + rank) * kArMax + i] = rc.red[i];
    }
    __syncthreads();
    if ((int)threadIdx.x < P) {
        __threadfence_system();
        unsigned long long *fl = reinterpret_cast<unsigned long long *>(pc.p[threadIdx.x] + kCbArFlags);
        st_release_sys(fl + par * 16 + rank, seq);
        const unsigned long long *mine = reinterpret_cast<const unsigned long long *>(pc.p[rank] + kCbArFlags);
        long long spins = 0;
        while (ld_acquire_sys(mine + par * 16 + threadIdx.x) < seq) {
            if (++spins > kSpinLimit) { rc.I[I_BREAKDOWN] = 1; break; }
        }
    }
    __syncthreads();
    const double *inbox = pc.p[rank] + kCbArInbox + (size_t)par * 16 * kArMax;
    if ((int)threadIdx.x < K) {
        double sum = 0.0;
        for (int r = 0; r < P; ++r) sum += __ldcg(inbox + (size_t)r * kArMax + threadIdx.x);
        rc.red[threadIdx.x] = sum;
    }
    if (threadIdx.x == 0) pc.ar_seq = seq;
    __syncthreads();
}

// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialisation attribute
// may start while its predecessor in the stream is still running; griddep_wait() blocks until the predecessor
// has completed and its memory is visible, griddep_launch() allows the successor to be scheduled.  Both are
// no-ops for kernels launched the ordinary way.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }


// ------------------------------------------------------------------------
// 5-point operator arithmetic.  OPK selects the reference's rounding order.
//   l = x(i-1), r = x(i+1), dn = x(idx+n) (next line), up = x(idx-n).
//   missing neighbours are passed as 0.0 (adding/subtracting 0.0 is exact, so
//   this reproduces every edge/corner formula of poisson.f90:47-76).
// ------------------------------------------------------------------------
// KL_OP_ANISO5: ex = eps_x, ey = eps_y, cc = 2(eps_x + eps_y) ; KL_OP_STENCIL5: ex = wl, ey = wd, cc = c and the two
// weights of the other side, exr = wr, eyu = wu (op_coef)
struct OpCoef {
    double ex, ey, cc;
    double exr, eyu;
};
inline OpCoef op_coef(const kl_operator_t *op) {
    if (op->kind == KL_OP_STENCIL5) {
        const kl_stencil5_t *w = (const kl_stencil5_t *)op->user;
        return OpCoef{w->wl, w->wd, w->c, w->wr, w->wu};
    }
    return OpCoef{op->eps_x, op->eps_y, 2.0 * (op->eps_x + op->eps_y), 0.0, 0.0};
}
template <int OPK>
__device__ __forceinline__ double apply5(double c, double l, double r, double dn, double up,
                                         const OpCoef &k) {
    if (OPK == KL_OP_POISSON5) {
        // poisson.f90:42  4*x - 1*(((x(idx-1)+x(idx+1))+x(idx+n))+x(idx-n))
        return 4.0 * c - (((l + r) + dn) + up);
    } else if (OPK == KL_OP_POISSON5_BRANCHY) {
        // poisson.f90:88-92  ((((4x - x(idx-1)) - x(idx+1)) - x(idx-n)) - x(idx+n))
        return (((4.0 * c - l) - r) - up) - dn;
    } else if (OPK == KL_OP_STENCIL5) {
        // krylov_b200.h kl_stencil5_t (the order of k_aniso_var)
        double s = fma(k.ex, l, k.exr * r), t = fma(k.ey, dn, k.eyu * up);
        return fma(k.cc, c, -(s + t));
    } else {
        double sx = l + r, sy = dn + up;
        double t = fma(k.ex, sx, k.ey * sy);
        return fma(k.cc, c, -t);
    }
}

// the same with the operator chosen at run time (generic, non-TMA kernel: small and odd grids, KL_OPT_TMA = 0).
// S5: KL_OP_STENCIL5, chosen at compile time -- its functors are wrapped in S5<F> (launch_stencil), so that the
// generic kernels of the other operators carry no fourth branch (it cost them registers and spills)
template <bool S5 = false>
__device__ __forceinline__ double apply5_rt(int opk, double c, double l, double r, double dn, double up, const OpCoef &k) {
    if (S5) return apply5<KL_OP_STENCIL5>(c, l, r, dn, up, k);
    if (opk == KL_OP_POISSON5) return apply5<KL_OP_POISSON5>(c, l, r, dn, up, k);
    if (opk == KL_OP_POISSON5_BRANCHY) return apply5<KL_OP_POISSON5_BRANCHY>(c, l, r, dn, up, k);
    return apply5<KL_OP_ANISO5>(c, l, r, dn, up, k);
}

// ------------------------------------------------------------------------
// Marching stencil kernel framework.
//
// A functor F describes a point-wise "input field" u (evaluated on the fly from
// NIN arrays, e.g. u = r/d or u = z + beta*p), the kernel applies the 5-point
// operator to u and hands (u, A u) to F::store, which writes outputs and
// accumulates up to NRED reductions.  Each thread owns VEC adjacent columns and
// marches down `rows` lines keeping three lines of u in registers, so every
// input element is loaded from L2/HBM once per block (plus 2 halo lines per
// `rows`).  Left/right neighbours come from warp shuffles; warp-edge lanes
// evaluate one extra scalar.
//
// Multi-GPU: lo/hi are the neighbour ranks' boundary lines of the NIN input
// arrays (nullptr at the global boundary => zero Dirichlet).
// ------------------------------------------------------------------------
// CTA tiling in the march direction.  blockIdx.y < gy_main: the regular tiles, `rows` lines on average, with the
// heights staggered in a period of four (h[0..3], prefix sums p[0..3], 4*rows per period) when stagger is on --
// CTAs that start together then finish at four different times, later generations mix further, and the memory
// system sees a steady stream instead of waves that start and drain in lockstep (measured time line:
// profiles/r02_cta_timeline.md).  The CTAs behind them (scheduled last) own `rows_tail` lines each: small tiles
// at the end of the grid shorten the kernel's tail.
struct Geo {
    int nx, ny, rows;
    int gy_main, rows_tail, main_end;
    int h0, h1, h2, h3;       // staggered heights of a period (scalars, not arrays: a run-time index into a kernel
    int p1, p2, p3;           // parameter makes the compiler copy the whole struct to local memory) ; prefix sums
    int reverse;              // 1: the tiling is mirrored, so the CTAs scheduled FIRST work on the LAST lines
    int gx, gy;               // strips x line bands = tiles (the TMA kernel's persistent CTAs loop over them)
};
// `reverse`: consecutive kernels of an iteration stream the same vectors (CG: K1 reads r, p ; K2 reads r, p again ;
// the next K1 reads the r that K2 wrote).  When a kernel starts where its predecessor stopped, the lines the
// predecessor touched last are still in the 126 MB L2 -- on the 268 MB-per-vector slabs of the 8-GPU strong-scaling
// run that is a tenth of the traffic; on 2 GB vectors it is noise.
__device__ __forceinline__ void tile_lines(const Geo &g, int by, int &j0, int &j1) {
    if (by < g.gy_main) {
        const int k = by & 3;
        const int pk = k == 0 ? 0 : (k == 1 ? g.p1 : (k == 2 ? g.p2 : g.p3));
        const int hk = k == 0 ? g.h0 : (k == 1 ? g.h1 : (k == 2 ? g.h2 : g.h3));
        j0 = (by >> 2) * (4 * g.rows) + pk;
        j1 = min(j0 + hk, g.main_end);
    } else {
        j0 = g.main_end + (by - g.gy_main) * g.rows_tail;
        j1 = min(j0 + g.rows_tail, g.ny);
    }
    if (g.reverse) {
        const int t = j0;
        j0 = g.ny - j1;
        j1 = g.ny - t;
    }
}

template <int NIN_, int NRED_>
struct StencilBase {
    static constexpr int NIN = NIN_;
    static constexpr int NRED = NRED_;
    // kPush: store() takes a trailing `int edge` (bit 0: the points lie on the slab's first line, bit 1: on its
    // last line) and may push those lines into the neighbour ranks' halo slots (multi-GPU, see kCbPush).
    static constexpr bool kPush = false;
    // kLateWait: nothing the kernel reads before its first store() is produced by the kernel launched just before
    // it (inputs, halo lines, the gate and what init() reads are older), so under programmatic dependent launch
    // the whole prologue -- barrier setup, the first TMA stages, the first lines of u -- overlaps the
    // predecessor's tail; late_init() then reads the predecessor's scalars.
    static constexpr bool kLateWait = false;
    // kReverse: march the grid from its last lines to its first (see Geo::reverse)
    static constexpr bool kReverse = false;
    // kS5: the generic kernel applies KL_OP_STENCIL5 (set by the S5<F> wrapper only)
    static constexpr bool kS5 = false;
    __device__ __forceinline__ void late_init() {}
    const double *in[NIN_];
    const double *lo[NIN_];
    const double *hi[NIN_];
    const int *flags;
    int step;         // gating: run iff flags[I_CONV_AT] < 0 (or == step when run_on_conv)
    int run_on_conv;
    OpCoef coef;
    __device__ __forceinline__ bool skip() const {
        if (!flags) return false;
        int ca = flags[I_CONV_AT];
        return !(ca < 0 || (run_on_conv && ca == step));
    }
};

// KL_OP_STENCIL5 on the generic kernel: the functor F with the operator fixed at compile time (apply5_rt<true>)
template <class F>
struct S5 : F {
    static constexpr bool kS5 = true;
};

constexpr int kStencilThreads = 128;

// Functor contract (see kl_functors.cuh):
//   double point(const double (&v)[NIN]) const      u at one grid point from the NIN raw inputs
//   template<int VEC> void store(size_t idx, const double (&raw)[NIN][VEC],
//                                const double (&cu)[VEC], const double (&au)[VEC], double *acc) const
// The kernel owns all loads: raw input lines are fetched kPf lines ahead of their
// use (software pipeline in registers) so that each thread keeps several
// independent 16-byte loads in flight; point() runs when a line is consumed.
constexpr int kPf = 2;   // prefetch distance in grid lines

template <class F, int VEC>
__global__ void __launch_bounds__(kStencilThreads)
k_stencil(const F f_in, const Geo g, const RedCtl rc, const PostAny post, const int fuse_post, const int opk) {
    griddep_wait();
    griddep_launch();
    if (f_in.skip()) return;
    F f = f_in;
    f.init();
    f.late_init();
    constexpr int NIN = F::NIN;
    constexpr int NRED = F::NRED;
    constexpr int NR = NRED > 0 ? NRED : 1;
    const int lane = threadIdx.x & 31;
    const int i0 = (blockIdx.x * kStencilThreads + threadIdx.x) * VEC;
    const bool act = i0 < g.nx;
    const bool has_l = act && lane == 0 && i0 > 0;
    const bool has_r = act && lane == 31 && i0 + VEC < g.nx;
    int j0, j1;
    tile_lines(g, blockIdx.y, j0, j1);
    double acc[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) acc[k] = 0.0;

    struct Raw {
        double c[NIN][VEC];
        double l[NIN], r[NIN];
        bool ok;
    };
    // raw loads of line j (may be a halo line or outside the domain)
    auto load_raw = [&](int j, Raw &R) {
        const double *rp[NIN];
        bool ok = act && j <= j1;
        if (ok) {
            if (j < 0) {
                ok = f.lo[0] != nullptr;
#pragma unroll
                for (int a = 0; a < NIN; ++a) rp[a] = f.lo[a];
            } else if (j >= g.ny) {
                ok = f.hi[0] != nullptr;
#pragma unroll
                for (int a = 0; a < NIN; ++a) rp[a] = f.hi[a];
            } else {
#pragma unroll
                for (int a = 0; a < NIN; ++a) rp[a] = f.in[a] + (size_t)j * g.nx;
            }
        }
        R.ok = ok;
#pragma unroll
        for (int a = 0; a < NIN; ++a) {
            if (ok) {
                if (VEC == 2) {
                    double2 t = ldg2(rp[a] + i0);
                    R.c[a][0] = t.x;
                    R.c[a][VEC - 1] = t.y;
                } else {
                    R.c[a][0] = __ldg(rp[a] + i0);
                }
            } else {
                R.c[a][0] = 0.0;
                R.c[a][VEC - 1] = 0.0;
            }
            R.l[a] = (ok && has_l) ? __ldg(rp[a] + i0 - 1) : 0.0;
            R.r[a] = (ok && has_r) ? __ldg(rp[a] + i0 + VEC) : 0.0;
        }
    };
    // u of a line from its raw inputs (+ the two warp-edge neighbours)
    auto compute = [&](const Raw &R, double (&u)[VEC], double &ul, double &ur) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            double t[NIN];
#pragma unroll
            for (int a = 0; a < NIN; ++a) t[a] = R.c[a][v];
            u[v] = R.ok ? f.point(t) : 0.0;
        }
        ul = (R.ok && has_l) ? f.point(R.l) : 0.0;
        ur = (R.ok && has_r) ? f.point(R.r) : 0.0;
    };

    Raw rawA, rawB, rawCu, rawDn;
    double up[VEC], cu[VEC], dn[VEC], cl, cr, dl, dr, tl, tr;
    {
        Raw t;
        load_raw(j0 - 1, t);
        load_raw(j0, rawCu);
        load_raw(j0 + 1, rawA);
        load_raw(j0 + 2, rawB);
        compute(t, up, tl, tr);
        compute(rawCu, cu, cl, cr);
    }
#pragma unroll 2
    for (int j = j0; j < j1; ++j) {
        Raw rawN;
        load_raw(j + 1 + kPf, rawN);          // prefetch, consumed kPf lines later
        compute(rawA, dn, dl, dr);
        rawDn = rawA;
        double l = __shfl_up_sync(0xffffffffu, cu[VEC - 1], 1);
        double r = __shfl_down_sync(0xffffffffu, cu[0], 1);
        if (lane == 0) l = cl;
        if (lane == 31) r = cr;
        if (act) {
            double au[VEC];
            if (VEC == 1) {
                au[0] = apply5_rt<F::kS5>(opk, cu[0], l, r, dn[0], up[0], f.coef);
            } else {
                au[0] = apply5_rt<F::kS5>(opk, cu[0], l, cu[VEC - 1], dn[0], up[0], f.coef);
                au[VEC - 1] = apply5_rt<F::kS5>(opk, cu[VEC - 1], cu[0], r, dn[VEC - 1], up[VEC - 1], f.coef);
            }
            if constexpr (F::kPush)
                f.template store<VEC>((size_t)j * g.nx + i0, rawCu.c, cu, au, acc, (j == 0 ? 1 : 0) | (j == g.ny - 1 ? 2 : 0));
            else
                f.template store<VEC>((size_t)j * g.nx + i0, rawCu.c, cu, au, acc);
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            up[v] = cu[v];
            cu[v] = dn[v];
        }
        cl = dl;
        cr = dr;
        rawCu = rawDn;
        rawA = rawB;
        rawB = rawN;
    }
    if (NRED > 0) {
        __shared__ double sm[NR * (kStencilThreads / 32)];
        __shared__ int s_flag;
        block_sum<NR, kStencilThreads>(acc, sm);
        const unsigned nb = gridDim.x * gridDim.y, bid = blockIdx.y * gridDim.x + blockIdx.x;
        if (grid_sum<NR, kStencilThreads>(acc, rc, nb, bid, &s_flag, sm)) {
            if (rc.peer) peer_allreduce_block<NR>(rc);
            if (fuse_post && threadIdx.x == 0) post.run();
        }
    }
}

// ------------------------------------------------------------------------
// Point-wise kernel framework: grid-stride over VEC-wide chunks, UNR chunks
// per thread per trip.  F::elem<VEC>(idx, acc) loads, computes and stores.
// ------------------------------------------------------------------------
constexpr int kPwThreads = 256;

// (min 3 resident blocks per SM = at most 85 registers: PBiUpdate reached 108 once the run-time post dispatch and
// the parallel final reduction were inlined into its tail, i.e. 2 blocks per SM, and lost a quarter of its bandwidth)
template <class F, int VEC>
__global__ void __launch_bounds__(kPwThreads, 3)
k_pointwise(const F f_in, const size_t n, const RedCtl rc, const PostAny post, const int fuse_post) {
    griddep_wait();
    if (f_in.skip()) return;
    F f = f_in;
    f.init();
    constexpr int NRED = F::NRED;
    double acc[NRED > 0 ? NRED : 1];
#pragma unroll
    for (int k = 0; k < (NRED > 0 ? NRED : 1); ++k) acc[k] = 0.0;
    const size_t nchunk = n / VEC;
    const size_t stride = (size_t)gridDim.x * kPwThreads;
#pragma unroll 4
    for (size_t c = (size_t)blockIdx.x * kPwThreads + threadIdx.x; c < nchunk; c += stride)
        f.template elem<VEC>(c * VEC, acc);
    if (NRED > 0) {
        __shared__ double sm[(NRED > 0 ? NRED : 1) * (kPwThreads / 32)];
        __shared__ int s_flag;
        block_sum<(NRED > 0 ? NRED : 1), kPwThreads>(acc, sm);
        if (grid_sum<(NRED > 0 ? NRED : 1), kPwThreads>(acc, rc, gridDim.x, blockIdx.x, &s_flag, sm)) {
            if (rc.peer) peer_allreduce_block<(NRED > 0 ? NRED : 1)>(rc);
            if (fuse_post && threadIdx.x == 0) post.run();
        }
    }
}

template <int NRED_>
struct PwBase {
    static constexpr int NRED = NRED_;
    const int *flags;
    int step;
    int run_on_conv;
    __device__ __forceinline__ bool skip() const {
        if (!flags) return false;
        int ca = flags[I_CONV_AT];
        return !(ca < 0 || (run_on_conv && ca == step));
    }
};


// post functor launched on its own (multi-GPU: after the all-reduce)
// red / red_src: the post functors read S_RED[0]; a kernel that reduces several sums (the Chebyshev chains keep
// both z.z and r.z so that their inner loop needs no selects) names the one to use
static __global__ void k_post(const PostAny post, const int *flags, const int step, const int run_on_conv,
                              double *red = nullptr, const int red_src = 0) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        if (flags) {   // same gate as the kernel whose sums it consumes
            const int ca = flags[I_CONV_AT];
            if (!(ca < 0 || (run_on_conv && ca == step))) return;
        }
        if (red && red_src) red[0] = red[red_src];
        post.run();
    }
}

// ------------------------------------------------------------------------
// launch helpers (host)
// ------------------------------------------------------------------------
inline RedCtl redctl(Ctx *c) { return RedCtl{c->d_partials, c->d_counter, c->d_S + S_RED, nullptr, c->d_I}; }

// Launch with or without the programmatic-stream-serialisation attribute.  ONLY for kernels that execute
// griddep_wait() before they read anything a predecessor wrote AND before any early exit (a grid that returns
// without waiting would let its successor overtake the grid before it).  Inside a PdlScope (a solver's step loop on
// one GPU) every such launch overlaps its launch latency, CTA scheduling and barrier set-up with the predecessor's
// tail: on the L2-resident problems (C1, 300^2) an Arnoldi step is five dependent ~5 us kernels and the launch gaps
// were a third of it.
struct PdlScope {
    Ctx *c;
    bool on;
    PdlScope(Ctx *c_, bool on_) : c(c_), on(on_) { if (on) ++c->pdl_scope; }
    ~PdlScope() { if (on) --c->pdl_scope; }
};
template <class... KArgs, class... Args>
inline cudaError_t launch_k(Ctx *c, bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                            Args &&...args) {
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = c->stream;
    cfg.attrs = at;
    cfg.numAttrs = ((pdl || c->pdl_scope > 0) && c->opt_pdl) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
// Reducing kernel on several GPUs with NVLink peer memory: the kernel's last block does the all-reduce and runs
// the post functor itself.  Returns true when that path is taken (then finish_reduction must not be called).
inline bool redctl_inline_allreduce(Ctx *c, RedCtl &rc, int nred) {
    if (c->nranks == 1 || !c->peer_ok || !c->d_peerctl || !c->opt_inline_ar || nred > kArMax) return false;
    rc.peer = c->d_peerctl;
    return true;
}

inline int stencil_rows(int nx, int ny, int vec) {
    // aim for >= ~8 blocks per SM, between 8 and 64 lines per block
    long gx = (nx + kStencilThreads * vec - 1) / (kStencilThreads * vec);
    long want = (long)kNumSM * 8;
    long rows = ((long)ny * gx + want - 1) / want;
    if (rows < 8) rows = 8;
    if (rows > 64) rows = 64;
    if (rows > ny) rows = ny;
    return (int)rows;
}

// after a reducing kernel: single GPU => post already ran fused; multi GPU =>
// all-reduce the local sums and run the post functor in its own kernel.
template <class Post>
inline int finish_reduction(Ctx *c, int nred, const Post &post, const int *flags = nullptr, int step = 0,
                            int run_on_conv = 0, int red_src = 0) {
    if (c->nranks > 1) {
        KL_TRY(comm_allreduce(c, c->d_S + S_RED, nred));
        k_post<<<1, 32, 0, c->stream>>>(to_any(post), flags, step, run_on_conv, c->d_S + S_RED, red_src);
        c->stats.kernel_launches++;
    }
    return KL_OK;
}

}  // namespace kl
#include "kl_stencil_tma.cuh"
namespace kl {

// CTA geometry: many short CTAs (8-64 grid lines each, >= ~8 CTAs per SM).  For these memory-bound kernels
// the tail of a partially filled last wave is self-correcting (the remaining CTAs get the whole HBM
// bandwidth), while few long CTAs load-balance badly: a "whole waves" geometry measured 8 % slower on the
// 8-GPU strong-scaling case (2048 local lines), so the simple rule stays.  `resident` is unused for now.
// persistent: the caller launches min(tiles, resident) CTAs that loop over the tiles, so the number of tiles is not
// bounded by the reduction buffer (one partial per CTA)
inline bool stencil_geometry(int nx, int ny, int strip, long resident, Geo *g, dim3 *grid, int rows_opt = 0,
                             int tail_opt = -1, int stagger = 1, bool persistent = false) {
    const long gx = (nx + strip - 1) / strip;
    if (gx > kMaxBlocks) return false;
    // Wide grids (>= 32 strips): ~28 CTAs per SM.  A CTA lives ~100 us there, and the kernel ends with a ragged
    // tail of about a third of that; on the 2048-line slab of the 8-GPU strong-scaling run 32-line CTAs (4224 CTAs)
    // measured 3 % faster per iteration than 64-line ones, while below 32 lines the per-CTA overhead and the two
    // halo lines per CTA cost more than the tail (scripts/slab_sweep.py, DESIGN.md section 6).
    const long want = (long)kNumSM * (gx >= 32 ? 16 : 8);     // (with the tapered tail, 57-line tiles measured 1 % faster
                                                               // than 33-line ones on the 2048-line slab of the 8-GPU run)
    long rows = ((long)ny * gx + want - 1) / want;
    if (rows < 8) rows = 8;
    if (rows > 128) rows = 128;            // 16384^2 on one GPU: 128-line tiles with a 32-line tail measured 2 % faster
    if (rows_opt > 0) rows = rows_opt;     // than 64 / 16 (scripts/slab_sweep2.py) ; KL_OPT_STENCIL_ROWS overrides
    if (rows > ny) rows = ny;
    long gy = (ny + rows - 1) / rows;
    // tapered tail (KL_OPT_STENCIL_TAIL: -1 auto, 0 off, > 0 lines per tail CTA): the last half wave of CTAs gets
    // tiles of a quarter of the height, so that the CTAs that finish last carry little work
    long rt = tail_opt < 0 ? (rows >= 32 ? rows / 4 : 0) : tail_opt;
    long tail_lines = 0, gy_tail = 0;
    const bool multiwave = resident > 0 && gx * gy > 2 * resident;
    if (rt > 0 && rt < rows && multiwave) {
        long tl = (resident / 2 + gx - 1) / gx * rows;           // lines covered by half a wave of full tiles
        if (tl > ny / 4) tl = ny / 4;
        tail_lines = tl;
    }
    // staggered heights 5/8, 7/8, 9/8, 11/8 of `rows` (KL_OPT_STENCIL_STAGGER)
    const bool stag = stagger && multiwave && rows >= 16;
    long h[4], p[4];
    for (int k = 0; k < 4; ++k) h[k] = stag ? rows * (5 + 2 * k) / 8 : rows;
    h[3] = 4 * rows - h[0] - h[1] - h[2];
    p[0] = 0;
    for (int k = 1; k < 4; ++k) p[k] = p[k - 1] + h[k - 1];
    auto count_main = [&](long main_end) {      // tiles needed to cover [0, main_end)
        long full = main_end / (4 * rows), rem = main_end - full * 4 * rows, n = 4 * full;
        for (int k = 0; k < 4 && rem > p[k]; ++k) ++n;
        return n;
    };
    long main_end = ny - tail_lines;
    long gy_main = count_main(main_end);
    if (tail_lines > 0) gy_tail = (tail_lines + rt - 1) / rt;
    if (!persistent && gx * (gy_main + gy_tail) > kMaxBlocks) {   // the deterministic reduction keeps one partial per CTA
        const long max_gy = kMaxBlocks / gx;
        rows = (ny + max_gy - 1) / max_gy;
        for (int k = 0; k < 4; ++k) { h[k] = rows; p[k] = k * rows; }
        main_end = ny;
        gy_main = (ny + rows - 1) / rows;
        gy_tail = 0;
        rt = 0;
    }
    g->nx = nx; g->ny = ny; g->rows = (int)rows;
    g->gy_main = (int)gy_main;
    g->rows_tail = (int)(gy_tail > 0 ? rt : rows);
    g->main_end = (int)main_end;
    g->gx = (int)gx;
    g->gy = (int)(gy_main + gy_tail);
    g->h0 = (int)h[0]; g->h1 = (int)h[1]; g->h2 = (int)h[2]; g->h3 = (int)h[3];
    g->p1 = (int)p[1]; g->p2 = (int)p[2]; g->p3 = (int)p[3];
    *grid = dim3((unsigned)gx, (unsigned)(gy_main + gy_tail));
    return true;
}

// pdl: launch with the programmatic-stream-serialisation attribute (the kernel's own griddep_wait() orders it
// after its predecessor; only for kernels that follow another k_stencil_tma / k_pointwise launch in the stream)
template <class F, class Post>
inline int launch_stencil(Ctx *c, const kl_operator_t *op, F f, int nx, int ny, const Post &post, bool pdl = false) {
    const int vec = (nx % 2 == 0) ? 2 : 1;
    const bool tma = c->opt_tma && vec == 2 && nx >= 64;
    // KL_OP_STENCIL5 runs the generic kernel with one column per thread only (S5<F>, VEC = 1: half the instantiations)
    const int strip = tma ? kTmaStrip : kStencilThreads * (op->kind == KL_OP_STENCIL5 ? 1 : vec);
    Geo g{};
    g.nx = nx; g.ny = ny;
    const int reverse = (F::kReverse && c->opt_reverse) ? 1 : 0;
    dim3 grid;
    f.coef = op_coef(op);
    RedCtl rc = redctl(c);
    const bool inl = F::NRED > 0 && redctl_inline_allreduce(c, rc, F::NRED);
    const int fuse = c->nranks == 1 || inl;
    const PostAny pa = to_any(post);
    const int opk = op->kind;
    TMaps<F::NIN> tm;
    if (tma) {
        for (int a = 0; a < F::NIN; ++a) KL_TRY(tmap_encode(c, &tm.m[a], f.in[a], nx, ny));
    }
    constexpr size_t smem = tma_smem_bytes<F::NIN>();
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kStencilThreads);
    cfg.stream = c->stream;
    cfg.attrs = at;
    cfg.numAttrs = ((pdl || c->pdl_scope > 0) && c->opt_pdl) ? 1 : 0;
    // the opt-in for > 48 KB of dynamic shared memory and the occupancy are per device (a process may hold
    // handles on several devices)
#define KL_ST_GEO(KERNEL, SMEM) KL_ST_GEO2(KERNEL, SMEM, false)
#define KL_ST_GEO2(KERNEL, SMEM, PERSIST)                                                           \
    {                                                                                               \
        static int occ[kMaxDevices] = {};                                                           \
        int &oc = occ[c->device % kMaxDevices];                                                     \
        if (!oc) {                                                                                  \
            if (SMEM > 0)                                                                           \
                cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM)); \
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&oc, KERNEL, kStencilThreads, SMEM) != cudaSuccess || \
                oc < 1)                                                                             \
                oc = 4;                                                                             \
        }                                                                                           \
        if (!stencil_geometry(nx, ny, strip, (long)oc * kNumSM, &g, &grid, c->opt_stencil_rows, c->opt_stencil_tail, c->opt_stencil_stagger, PERSIST)) \
            return c->fail(KL_ERR_UNSUPPORTED, "grid too wide for the reduction buffer");           \
        g.reverse = reverse;                                                                        \
        if (PERSIST) {   /* persistent CTAs: as many as are resident at once (KL_OPT_PERSIST_OCC CTAs per SM) */ \
            long res = (long)((c->opt_persist_occ > 0 && c->opt_persist_occ < oc) ? c->opt_persist_occ : oc) * kNumSM; \
            long tiles = (long)grid.x * grid.y;                                                     \
            if (!c->opt_persistent) res = tiles;                                                    \
            if (res > kMaxBlocks) res = kMaxBlocks;                                                 \
            /* balanced: every CTA gets the same number of tiles (+-1), so that they all finish together */ \
            const long rounds = (tiles + res - 1) / res;                                            \
            grid = dim3((unsigned)((tiles + rounds - 1) / rounds));                                 \
        }                                                                                           \
        cfg.gridDim = grid;                                                                         \
        cfg.dynamicSmemBytes = SMEM;                                                                \
    }
    if (opk != KL_OP_POISSON5 && opk != KL_OP_POISSON5_BRANCHY && opk != KL_OP_ANISO5 && opk != KL_OP_STENCIL5)
        return c->fail(KL_ERR_INVALID, "launch_stencil: not a built-in operator");
    // the TMA kernel is specialised per operator (its inner loop is the hot path); the generic kernel takes it as
    // a run-time argument
#define KL_ST_TMA(OPK)                                                                              \
    {                                                                                               \
        KL_ST_GEO2((k_stencil_tma<F, OPK>), smem, true)                                             \
        KL_CUDA(c, cudaLaunchKernelEx(&cfg, k_stencil_tma<F, OPK>, f, g, rc, pa, fuse, tm));        \
    }
    if (tma) {
        if (opk == KL_OP_POISSON5) KL_ST_TMA(KL_OP_POISSON5)
        else if (opk == KL_OP_POISSON5_BRANCHY) KL_ST_TMA(KL_OP_POISSON5_BRANCHY)
        else if (opk == KL_OP_STENCIL5) KL_ST_TMA(KL_OP_STENCIL5)
        else KL_ST_TMA(KL_OP_ANISO5)
    } else if (opk == KL_OP_STENCIL5) {
        S5<F> f5;
        static_cast<F &>(f5) = f;
        KL_ST_GEO((k_stencil<S5<F>, 1>), 0)
        KL_CUDA(c, cudaLaunchKernelEx(&cfg, k_stencil<S5<F>, 1>, f5, g, rc, pa, fuse, opk));
    } else if (vec == 2) {
        KL_ST_GEO((k_stencil<F, 2>), 0)
        KL_CUDA(c, cudaLaunchKernelEx(&cfg, k_stencil<F, 2>, f, g, rc, pa, fuse, opk));
    } else {
        KL_ST_GEO((k_stencil<F, 1>), 0)
        KL_CUDA(c, cudaLaunchKernelEx(&cfg, k_stencil<F, 1>, f, g, rc, pa, fuse, opk));
    }
#undef KL_ST_TMA
#undef KL_ST_GEO
#undef KL_ST_GEO2
    c->stats.kernel_launches++;
    if (F::NRED > 0 && !inl) return finish_reduction(c, F::NRED, post, f.flags, f.step, f.run_on_conv);
    return KL_OK;
}

inline int pw_grid(size_t nchunk) {
    size_t b = (nchunk + kPwThreads * 4 - 1) / (kPwThreads * 4);
    size_t cap = (size_t)kNumSM * 8;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

template <class F, class Post>
inline int launch_pointwise(Ctx *c, F f, size_t n, const Post &post) {
    RedCtl rc = redctl(c);
    const bool inl = F::NRED > 0 && redctl_inline_allreduce(c, rc, F::NRED);
    const int fuse = c->nranks == 1 || inl;
    const PostAny pa = to_any(post);
    if (n % 2 == 0)
        KL_CUDA(c, launch_k(c, false, k_pointwise<F, 2>, dim3(pw_grid(n / 2)), dim3(kPwThreads), 0, f, n, rc, pa, fuse));
    else
        KL_CUDA(c, launch_k(c, false, k_pointwise<F, 1>, dim3(pw_grid(n)), dim3(kPwThreads), 0, f, n, rc, pa, fuse));
    c->stats.kernel_launches++;
    if (F::NRED > 0 && !inl) return finish_reduction(c, F::NRED, post, f.flags, f.step, f.run_on_conv);
    return KL_OK;
}

}  // namespace kl
