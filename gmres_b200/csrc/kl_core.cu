// kl_core.cu -- handle lifecycle, options, workspace, device vectors, NCCL plumbing.
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include <cuda.h>
#include <cudaTypedefs.h>

#include "kl_internal.cuh"

namespace kl {

Ctx::GraphEntry *graph_find(Ctx *c, const std::string &key) {
    for (auto &g : c->graphs)
        if (g.key == key) return &g;
    return nullptr;
}
void graph_clear(Ctx *c) {
    for (auto &g : c->graphs) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
}
int graph_begin(Ctx *c) {
    if (c->capturing) return c->fail(KL_ERR_INVALID, "nested graph capture");
    if (!c->cap_stream) KL_CUDA(c, cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
    c->saved_stream = c->stream;
    c->stream = c->cap_stream;
    cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed);
    if (e != cudaSuccess) {
        c->stream = c->saved_stream;
        return c->fail(KL_ERR_CUDA, "cudaStreamBeginCapture", e);
    }
    c->capturing = true;
    return KL_OK;
}
int graph_end(Ctx *c, const std::string &key, double bytes, long long launches, Ctx::GraphEntry **out) {
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    c->stream = c->saved_stream;
    c->capturing = false;
    if (e != cudaSuccess || !g) {
        cudaGetLastError();
        return c->fail(KL_ERR_CUDA, "cudaStreamEndCapture", e);
    }
    cudaGraphExec_t ex = nullptr;
    e = cudaGraphInstantiate(&ex, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return c->fail(KL_ERR_CUDA, "cudaGraphInstantiate", e);
    }
    if (c->graphs.size() >= 16) {      // small cache: the oldest entry goes
        cudaGraphExecDestroy(c->graphs.front().exec);
        c->graphs.erase(c->graphs.begin());
    }
    c->graphs.push_back(Ctx::GraphEntry{key, ex, bytes, launches});
    *out = &c->graphs.back();
    return KL_OK;
}

int ws_reserve(Ctx *c, size_t bytes) {
    if (bytes <= c->ws_bytes) return KL_OK;
    graph_clear(c);     // cached graphs hold addresses inside the old arena
    if (c->ws) {
        cudaStreamSynchronize(c->stream);
        cudaFree(c->ws);
        c->ws = nullptr;
        c->ws_bytes = 0;
    }
    cudaError_t e = cudaMalloc(&c->ws, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return c->fail(KL_ERR_ALLOC, "workspace cudaMalloc", e);
    }
    c->ws_bytes = bytes;
    return KL_OK;
}

// 2-D FP64 tensor maps (zero fill outside the tensor).  Descriptors are cached per handle, keyed by
// (base pointer, extents, k1, k2); cuTensorMapEncodeTiled is taken from the driver through the runtime so that
// libcuda is not a link-time dependency.
static int tmap_get(Ctx *c, CUtensorMap *out, const void *base, int key_nx, int key_ny, long long k1, long long k2,
                    cuuint64_t dim0, cuuint64_t dim1, cuuint64_t row_pitch_bytes, cuuint32_t box0, cuuint32_t box1,
                    CUtensorMapL2promotion l2, const char *what) {
    static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap size");
    for (auto &e : c->tmaps)
        if (e.base == base && e.nx == key_nx && e.ny == key_ny && e.k1 == k1 && e.k2 == k2) {
            memcpy(out, e.blob, sizeof(CUtensorMap));
            return KL_OK;
        }
    if (!c->encode_fn) {
        cudaDriverEntryPointQueryResult q;
        void *fn = nullptr;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
        if (e != cudaSuccess || !fn) return c->fail(KL_ERR_CUDA, "cuTensorMapEncodeTiled entry point", e);
        c->encode_fn = fn;
    }
    auto enc = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(c->encode_fn);
    cuuint64_t dims[2] = {dim0, dim1};
    cuuint64_t strides[1] = {row_pitch_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return c->fail(KL_ERR_CUDA, what);
    if (c->tmaps.size() >= 256) c->tmaps.clear();
    Ctx::TmapEntry e;
    e.base = base; e.nx = key_nx; e.ny = key_ny; e.k1 = k1; e.k2 = k2;
    memcpy(e.blob, out, sizeof(CUtensorMap));
    c->tmaps.push_back(e);
    return KL_OK;
}

// nx x ny grid (i fastest), box = 256 columns x kTmaSR lines (k_stencil_tma)
int tmap_encode(Ctx *c, CUtensorMap *out, const double *base, int nx, int ny) {
    return tmap_get(c, out, base, nx, ny, 0, 0, (cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)nx * sizeof(double),
                    kTmaBoxX, kTmaSR, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "cuTensorMapEncodeTiled failed");
}

// grid tensor map with an explicit box (chained stencil kernels, kl_chain_tma.cuh); key: k1 = box_x, k2 = box_y
int tmap_encode_box(Ctx *c, CUtensorMap *out, const double *base, int nx, int ny, int box_x, int box_y) {
    return tmap_get(c, out, base, nx, ny, box_x, box_y, (cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)nx * sizeof(double),
                    (cuuint32_t)box_x, (cuuint32_t)box_y, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    "cuTensorMapEncodeTiled (box) failed");
}

// Krylov basis V (n rows fastest, ncols_total columns, ld = ldv), box = 32*RM rows x nc columns (k_ts_tma).
// key: the ny field carries -nc so that it cannot collide with a grid map
static inline int ts_rm_host(int nc) { return nc <= 12 ? 8 : (nc <= 24 ? 4 : (nc <= 48 ? 2 : 1)); }
int tmap_encode_v(Ctx *c, CUtensorMap *out, const double *V, size_t n, size_t ldv, int ncols_total, int nc) {
    return tmap_get(c, out, V, (int)n, -nc, (long long)ldv, ncols_total, (cuuint64_t)n, (cuuint64_t)ncols_total,
                    (cuuint64_t)ldv * sizeof(double), (cuuint32_t)(32 * ts_rm_host(nc)), (cuuint32_t)nc,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "cuTensorMapEncodeTiled (V) failed");
}

void prof_reset(Ctx *c) {
    for (auto &r : c->prof_recs) { c->prof_pool.push_back(r.a); c->prof_pool.push_back(r.b); }
    c->prof_recs.clear();
    for (int i = 0; i < KL_PROFILE_CLASSES; ++i) {
        c->prof_ms[i] = 0; c->prof_launches[i] = 0; c->prof_bytes[i] = 0; c->prof_name[i] = nullptr;
    }
}
static cudaEvent_t prof_event(Ctx *c) {
    if (!c->prof_pool.empty()) { cudaEvent_t e = c->prof_pool.back(); c->prof_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
void prof_begin(Ctx *c, int cls, const char *name, double bytes) {
    Ctx::ProfRec r{cls, prof_event(c), prof_event(c)};
    c->prof_name[cls] = name;
    c->prof_bytes[cls] += bytes;
    c->prof_launches[cls] += 1;
    cudaEventRecord(r.a, c->stream);
    c->prof_recs.push_back(r);
}
void prof_end(Ctx *c) { cudaEventRecord(c->prof_recs.back().b, c->stream); }
void prof_resolve(Ctx *c) {
    for (auto &r : c->prof_recs) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) c->prof_ms[r.cls] += ms;
    }
    cudaGetLastError();
}

// ------------------------------------------------------------------------
// NCCL, loaded at run time (dlopen) so that the library has no link-time
// dependency on it: single-GPU users and CPU-only symbol checks never need it,
// and under torchrun the process-wide libnccl.so.2 that torch already loaded is
// the one that gets used.
// ------------------------------------------------------------------------
typedef struct { char internal[128]; } ncclUniqueId_t;
typedef void *ncclComm_p;
enum { kNcclFloat64 = 8, kNcclSum = 0 };
struct Nccl {
    void *lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId_t *) = nullptr;
    int (*CommInitRank)(ncclComm_p *, int, ncclUniqueId_t, int) = nullptr;
    int (*CommDestroy)(ncclComm_p) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_p, cudaStream_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;

static int nccl_load(std::string *err) {
    if (g_nccl.lib) return KL_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
    void *lib = nullptr;
    const char *env = getenv("KL_NCCL_LIB");
    if (env) lib = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
    for (int i = 0; !lib && names[i]; ++i) lib = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!lib) {
        if (err) *err = std::string("cannot dlopen libnccl.so.2: ") + dlerror();
        return KL_ERR_NCCL;
    }
#define KL_SYM(field, name)                                            \
    *(void **)(&g_nccl.field) = dlsym(lib, name);                      \
    if (!g_nccl.field) {                                               \
        if (err) *err = std::string("missing NCCL symbol ") + name;    \
        return KL_ERR_NCCL;                                            \
    }
    KL_SYM(GetUniqueId, "ncclGetUniqueId")
    KL_SYM(CommInitRank, "ncclCommInitRank")
    KL_SYM(CommDestroy, "ncclCommDestroy")
    KL_SYM(AllReduce, "ncclAllReduce")
    KL_SYM(AllGather, "ncclAllGather")
    KL_SYM(Send, "ncclSend")
    KL_SYM(Recv, "ncclRecv")
    KL_SYM(GroupStart, "ncclGroupStart")
    KL_SYM(GroupEnd, "ncclGroupEnd")
    KL_SYM(GetErrorString, "ncclGetErrorString")
#undef KL_SYM
    g_nccl.lib = lib;
    return KL_OK;
}

#define KL_NCCL(c, call)                                                                   \
    do {                                                                                   \
        int r__ = (call);                                                                  \
        if (r__ != 0) {                                                                    \
            (c)->err = std::string(#call ": ") + g_nccl.GetErrorString(r__);               \
            return KL_ERR_NCCL;                                                            \
        }                                                                                  \
    } while (0)

// ------------------------------------------------------------------------
// NVLink peer-memory collectives.  Every message on this path is latency-class
// (1-96 doubles per all-reduce, one grid line per halo), so what matters is the
// number of launches and round trips, not bandwidth.  Each rank owns a small
// communication buffer that all ranks of the node map through CUDA IPC:
//   all-reduce: every rank PUSHES its partial sums into every peer's inbox
//     (posted NVLink writes) and raises a sequence flag; one kernel then waits
//     for the P flags and sums the inbox in rank order -- same bits on every
//     rank, no broadcast needed.  One ~5 us kernel instead of an NCCL launch.
//   halo: each rank pushes its boundary lines straight into the neighbours'
//     halo buffers and waits for theirs.
// Buffers are double-buffered by sequence parity: a rank can be at most one
// collective ahead of a peer (it needs the peer's contribution to go further).
// If IPC mapping is not possible the NCCL path below is used instead.
// ------------------------------------------------------------------------
struct PeerPtrs {
    double *p[16];
};
__global__ void k_peer_allreduce(double *buf, const int count, PeerCtl *ctl, int *I) {
    const PeerCtl &pc = *ctl;
    const int rank = pc.rank, P = pc.nranks;
    const unsigned long long seq = pc.ar_seq + 1ull;    // sequence of EXECUTED all-reduces (see PeerCtl)
    const int par = (int)(seq & 1ull);
    // push my values into every rank's inbox (including my own)
    for (int t = threadIdx.x; t < count * P; t += blockDim.x) {
        const int q = t / count, i = t - q * count;
        pc.p[q][kCbArInbox + ((size_t)par * 16 + rank) * kArMax + i] = buf[i];
    }
    __syncthreads();
    if (threadIdx.x < P) {
        __threadfence_system();
        unsigned long long *fl = reinterpret_cast<unsigned long long *>(pc.p[threadIdx.x] + kCbArFlags);
        st_release_sys(fl + par * 16 + rank, seq);
    }
    // wait for every rank's contribution
    if (threadIdx.x < P) {
        const unsigned long long *fl = reinterpret_cast<const unsigned long long *>(pc.p[rank] + kCbArFlags);
        long long spins = 0;
        while (ld_acquire_sys(fl + par * 16 + threadIdx.x) < seq) {
            if (++spins > kSpinLimit) { I[I_BREAKDOWN] = 1; break; }
        }
    }
    __syncthreads();
    const double *inbox = pc.p[rank] + kCbArInbox + (size_t)par * 16 * kArMax;
    for (int i = threadIdx.x; i < count; i += blockDim.x) {
        double sum = 0.0;
        for (int r = 0; r < P; ++r) sum += __ldcg(inbox + (size_t)r * kArMax + i);
        buf[i] = sum;
    }
    if (threadIdx.x == 0) ctl->ar_seq = seq;
}

// Boundary lines of up to four slab vectors stored straight into the neighbours' PUSH slots (kCbPush) -- the
// set-up step of the "producer pushes" halo scheme (kl_cg.cu): no flags, the all-reduce of the next reducing
// kernel in the stream is the barrier.  block b = 2*v + dir ; dir 0: my first `count` doubles go to rank-1's
// hi slot, dir 1: my last ones to rank+1's lo slot.  src == nullptr pushes zeros.
struct PushArgs {
    const double *first[4], *last[4];
    int slot[4];
};
__global__ void k_push_lines(const PeerCtl *ctl, const PushArgs a, const int parity, const int count) {
    const int v = blockIdx.x >> 1, dir = blockIdx.x & 1;
    const int nb = dir == 0 ? ctl->rank - 1 : ctl->rank + 1;
    if (nb < 0 || nb >= ctl->nranks) return;
    const double *src = dir == 0 ? a.first[v] : a.last[v];
    double *dst = ctl->p[nb] + push_slot_off(parity, a.slot[v], 1 - dir);
    for (int i = threadIdx.x * 2; i < count; i += blockDim.x * 2) {
        double2 t = src ? *reinterpret_cast<const double2 *>(src + i) : make_double2(0.0, 0.0);
        *reinterpret_cast<double2 *>(dst + i) = t;
    }
    __threadfence_system();
}

// block b = 2*v + dir: dir 0 sends my first line of vector v to rank-1 (its "hi" halo) and waits for
// rank-1's last line (my "lo" halo); dir 1 the mirror image.
__global__ void k_peer_halo(const PeerPtrs pp, const int rank, const int P, const int nx,
                            const unsigned long long seq, const double *s0, const double *s1, const double *s2,
                            const double *s3, const double *e0, const double *e1, const double *e2, const double *e3,
                            int *I) {
    const int v = blockIdx.x >> 1, dir = blockIdx.x & 1;
    const int par = (int)(seq & 1ull);
    const double *first[4] = {s0, s1, s2, s3}, *last[4] = {e0, e1, e2, e3};
    const int nb = dir == 0 ? rank - 1 : rank + 1;
    if (nb < 0 || nb >= P) return;
    // my line goes into the neighbour's opposite-direction halo slot
    const double *src = dir == 0 ? first[v] : last[v];
    double *dst = pp.p[nb] + kCbHalo + (((size_t)par * 4 + v) * 2 + (1 - dir)) * kHaloNxCap;
    for (int i = threadIdx.x * 2; i < nx; i += blockDim.x * 2) {
        if (i + 1 < nx) *reinterpret_cast<double2 *>(dst + i) = *reinterpret_cast<const double2 *>(src + i);
        else dst[i] = src[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        unsigned long long *fl = reinterpret_cast<unsigned long long *>(pp.p[nb] + kCbHaloFlags);
        st_release_sys(fl + (par * 4 + v) * 2 + (1 - dir), seq);
        const unsigned long long *mine = reinterpret_cast<const unsigned long long *>(pp.p[rank] + kCbHaloFlags);
        long long spins = 0;
        while (ld_acquire_sys(mine + (par * 4 + v) * 2 + dir) < seq) {
            if (++spins > kSpinLimit) { I[I_BREAKDOWN] = 1; break; }
        }
    }
}

static PeerPtrs peer_ptrs(const Ctx *c) {
    PeerPtrs pp;
    for (int i = 0; i < 16; ++i) pp.p[i] = c->cb_peer[i];
    return pp;
}

int comm_allreduce(Ctx *c, double *d_buf, int count) {
    if (c->nranks == 1) return KL_OK;
    if (c->peer_ok && c->d_peerctl && count <= kArMax) {
        k_peer_allreduce<<<1, 256, 0, c->stream>>>(d_buf, count, c->d_peerctl, c->d_I);
        c->stats.kernel_launches++;
        return KL_OK;
    }
    KL_NCCL(c, g_nccl.AllReduce(d_buf, d_buf, (size_t)count, kNcclFloat64, kNcclSum,
                                (ncclComm_p)c->nccl_comm, c->stream));
    return KL_OK;
}

// Exchange the boundary lines of `nvec` slab vectors with the neighbour ranks.
// send_lo_rows[v] = this rank's first line, goes to rank-1's `hi` halo;
// send_hi_rows[v] = this rank's last line, goes to rank+1's `lo` halo.
int comm_halo_exchange(Ctx *c, const double *const *send_lo_rows, const double *const *send_hi_rows,
                       const double **lo_out, const double **hi_out, int nvec, int nx) {
    for (int a = 0; a < 4; ++a) lo_out[a] = hi_out[a] = nullptr;
    if (c->nranks == 1) return KL_OK;
    const bool has_lo = c->rank > 0, has_hi = c->rank < c->nranks - 1;
    if (c->peer_ok && nx <= kHaloNxCap && nx % 2 == 0) {
        ++c->halo_seq;
        const int par = (int)(c->halo_seq & 1ull);
        const double *s[4] = {nullptr, nullptr, nullptr, nullptr}, *e[4] = {nullptr, nullptr, nullptr, nullptr};
        for (int v = 0; v < nvec; ++v) {
            s[v] = send_lo_rows[v];
            e[v] = send_hi_rows[v];
            const double *base = c->cb_local + kCbHalo + ((size_t)par * 4 + v) * 2 * kHaloNxCap;
            lo_out[v] = has_lo ? base : nullptr;
            hi_out[v] = has_hi ? base + kHaloNxCap : nullptr;
        }
        k_peer_halo<<<2 * nvec, 256, 0, c->stream>>>(peer_ptrs(c), c->rank, c->nranks, nx, c->halo_seq, s[0],
                                                     s[1], s[2], s[3], e[0], e[1], e[2], e[3], c->d_I);
        c->stats.kernel_launches++;
        return KL_OK;
    }
    ncclComm_p comm = (ncclComm_p)c->nccl_comm;
    KL_NCCL(c, g_nccl.GroupStart());
    for (int v = 0; v < nvec; ++v) {
        double *rlo = c->d_halo + (size_t)(2 * v) * nx, *rhi = c->d_halo + (size_t)(2 * v + 1) * nx;
        lo_out[v] = has_lo ? rlo : nullptr;
        hi_out[v] = has_hi ? rhi : nullptr;
        if (has_lo) {
            KL_NCCL(c, g_nccl.Send(send_lo_rows[v], nx, kNcclFloat64, c->rank - 1, comm, c->stream));
            KL_NCCL(c, g_nccl.Recv(rlo, nx, kNcclFloat64, c->rank - 1, comm, c->stream));
        }
        if (has_hi) {
            KL_NCCL(c, g_nccl.Send(send_hi_rows[v], nx, kNcclFloat64, c->rank + 1, comm, c->stream));
            KL_NCCL(c, g_nccl.Recv(rhi, nx, kNcclFloat64, c->rank + 1, comm, c->stream));
        }
    }
    KL_NCCL(c, g_nccl.GroupEnd());
    return KL_OK;
}

// "Producer pushes" halo scheme: is it available (all ranks take the same decision)?  count = doubles per line.
bool comm_push_ok(const Ctx *c, int count) {
    return c->nranks > 1 && c->peer_ok && c->d_peerctl && c->opt_inline_ar && c->opt_push_halo &&
           count <= kHaloNxCap && count % 2 == 0;
}
// where the neighbours' lines of (parity, slot) arrive in MY buffer: lo = rank-1's last line, hi = rank+1's first
void comm_push_recv(const Ctx *c, int parity, int slot, const double **lo, const double **hi) {
    *lo = c->rank > 0 ? c->cb_local + push_slot_off(parity, slot, 0) : nullptr;
    *hi = c->rank < c->nranks - 1 ? c->cb_local + push_slot_off(parity, slot, 1) : nullptr;
}
// where MY first / last line of (parity, slot) has to be stored: rank-1's hi slot / rank+1's lo slot
void comm_push_send(const Ctx *c, int parity, int slot, double **first_dst, double **last_dst) {
    *first_dst = c->rank > 0 ? c->cb_peer[c->rank - 1] + push_slot_off(parity, slot, 1) : nullptr;
    *last_dst = c->rank < c->nranks - 1 ? c->cb_peer[c->rank + 1] + push_slot_off(parity, slot, 0) : nullptr;
}
int comm_push_lines(Ctx *c, int nvec, const double *const *first, const double *const *last, const int *slots,
                    int parity, int count) {
    if (nvec < 1 || nvec > 4) return c->fail(KL_ERR_INVALID, "comm_push_lines: 1..4 vectors");
    PushArgs a{};
    for (int v = 0; v < nvec; ++v) { a.first[v] = first[v]; a.last[v] = last[v]; a.slot[v] = slots[v]; }
    k_push_lines<<<2 * nvec, 256, 0, c->stream>>>(c->d_peerctl, a, parity, count);
    c->stats.kernel_launches++;
    return KL_OK;
}

// Map every rank's communication buffer into this process (CUDA IPC handles all-gathered over NCCL).
static int peer_setup(Ctx *c) {
    c->peer_ok = false;
    if (!c->opt_peer || c->nranks > 16 || getenv("KL_NO_PEER")) return KL_OK;
    if (cudaMalloc(&c->cb_local, kCbDoubles * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return KL_OK; }
    cudaMemset(c->cb_local, 0, kCbDoubles * sizeof(double));
    cudaIpcMemHandle_t mine;
    if (cudaIpcGetMemHandle(&mine, c->cb_local) != cudaSuccess) { cudaGetLastError(); return KL_OK; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    unsigned char *d_all = nullptr;
    if (cudaMalloc(&d_all, 64 * (size_t)c->nranks) != cudaSuccess) { cudaGetLastError(); return KL_OK; }
    cudaMemcpy(d_all + 64 * (size_t)c->rank, &mine, 64, cudaMemcpyHostToDevice);
    if (!g_nccl.AllGather) { cudaFree(d_all); return KL_OK; }
    int rc = g_nccl.AllGather(d_all + 64 * (size_t)c->rank, d_all, 64, 0 /* ncclInt8 */, (ncclComm_p)c->nccl_comm, c->stream);
    if (rc != 0 || cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); cudaFree(d_all); return KL_OK; }
    std::vector<cudaIpcMemHandle_t> all(c->nranks);
    cudaMemcpy(all.data(), d_all, 64 * (size_t)c->nranks, cudaMemcpyDeviceToHost);
    cudaFree(d_all);
    bool ok = true;
    for (int r = 0; r < c->nranks; ++r) {
        if (r == c->rank) { c->cb_peer[r] = c->cb_local; continue; }
        void *ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            ok = false;
            break;
        }
        c->cb_peer[r] = (double *)ptr;
    }
    // every rank must agree, otherwise some would wait on flags that never come
    double flag = ok ? 0.0 : 1.0, *d_flag = nullptr;
    cudaMalloc(&d_flag, sizeof(double));
    cudaMemcpy(d_flag, &flag, sizeof(double), cudaMemcpyHostToDevice);
    g_nccl.AllReduce(d_flag, d_flag, 1, kNcclFloat64, kNcclSum, (ncclComm_p)c->nccl_comm, c->stream);
    cudaStreamSynchronize(c->stream);
    cudaMemcpy(&flag, d_flag, sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(d_flag);
    c->peer_ok = (flag == 0.0);
    if (c->peer_ok) {
        PeerCtl pc;
        for (int r = 0; r < 16; ++r) pc.p[r] = c->cb_peer[r];
        pc.rank = c->rank;
        pc.nranks = c->nranks;
        pc.ar_seq = 0ull;
        if (cudaMalloc(&c->d_peerctl, sizeof(PeerCtl)) == cudaSuccess)
            cudaMemcpy(c->d_peerctl, &pc, sizeof(PeerCtl), cudaMemcpyHostToDevice);
        else { cudaGetLastError(); c->d_peerctl = nullptr; c->peer_ok = false; }
    }
    // KL_OPT_PEER may re-enable the peer path later only if EVERY rank mapped every buffer
    c->peer_mapped = c->peer_ok;
    return KL_OK;
}

}  // namespace kl

using namespace kl;

extern "C" {

int kl_version(void) { return KL_VERSION; }

int kl_create(kl_handle_t *h, int device) {
    if (!h) return KL_ERR_INVALID;
    *h = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return KL_ERR_CUDA;  // fail loudly: there is no CPU fallback
    }
    if (device < 0 || device >= ndev) return KL_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return KL_ERR_CUDA;
    Ctx *c = new Ctx();
    c->device = device;
    // experiment switches (same meaning as the options; options set later win)
    if (const char *e = getenv("KL_PDL")) c->opt_pdl = atoi(e) != 0;
    if (const char *e = getenv("KL_USE_GRAPH")) c->opt_use_graph = atoi(e) != 0;
    if (const char *e = getenv("KL_STENCIL_TAIL")) c->opt_stencil_tail = atoi(e);
    if (const char *e = getenv("KL_STENCIL_STAGGER")) c->opt_stencil_stagger = atoi(e) != 0;
    if (const char *e = getenv("KL_REVERSE")) c->opt_reverse = atoi(e) != 0;
    if (const char *e = getenv("KL_CG_ONEPASS")) c->opt_cg_onepass = atoi(e) < 0 ? -1 : std::min(atoi(e), 3);
    if (const char *e = getenv("KL_CG_GROUP")) c->opt_cg_group = std::max(2, std::min(atoi(e), 4));
    if (const char *e = getenv("KL_COOP")) c->opt_coop = atoi(e) != 0;
    if (const char *e = getenv("KL_PERSISTENT")) c->opt_persistent = atoi(e) != 0;
    if (const char *e = getenv("KL_PERSIST_OCC")) c->opt_persist_occ = atoi(e);
    if (const char *e = getenv("KL_TS_BLOCKS")) c->opt_ts_blocks = atoi(e);
    if (const char *e = getenv("KL_CHAIN_STEP_MIN")) c->opt_chain_step_min = atoll(e);
    if (const char *e = getenv("KL_CHAIN_ROWS_MIN")) c->opt_chain_rows_min = atoi(e);
    if (const char *e = getenv("KL_STENCIL_ROWS")) c->opt_stencil_rows = atoi(e);
    if (const char *e = getenv("KL_PUSH_HALO")) c->opt_push_halo = atoi(e) != 0;
    if (const char *e = getenv("KL_INLINE_ALLREDUCE")) c->opt_inline_ar = atoi(e) != 0;
    bool ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaMalloc(&c->d_S, sizeof(double) * S_COUNT) == cudaSuccess;
    ok = ok && cudaMalloc(&c->d_I, sizeof(int) * I_COUNT) == cudaSuccess;
    ok = ok && cudaMalloc(&c->d_partials, sizeof(double) * std::max((size_t)kMaxCols * 1024, (size_t)kMaxRed * kMaxBlocks)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->d_counter, sizeof(unsigned) * 128) == cudaSuccess;
    c->hist_cap = 1 << 20;
    ok = ok && cudaMalloc(&c->d_hist, sizeof(double) * c->hist_cap) == cudaSuccess;
    ok = ok && cudaMallocHost(&c->h_pinned, sizeof(double) * S_COUNT) == cudaSuccess;
    ok = ok && cudaMallocHost(&c->h_pinned_i, sizeof(int) * I_COUNT) == cudaSuccess;
    ok = ok && cudaEventCreate(&c->ev0) == cudaSuccess && cudaEventCreate(&c->ev1) == cudaSuccess;
    ok = ok && cudaEventCreate(&c->ev2) == cudaSuccess && cudaEventCreate(&c->ev3) == cudaSuccess;
    if (ok) {
        ok = cudaMemset(c->d_S, 0, sizeof(double) * S_COUNT) == cudaSuccess &&
             cudaMemset(c->d_I, 0, sizeof(int) * I_COUNT) == cudaSuccess &&
             cudaMemset(c->d_counter, 0, sizeof(unsigned) * 128) == cudaSuccess;
    }
    if (!ok) {
        cudaGetLastError();
        kl_destroy(c);
        return KL_ERR_ALLOC;
    }
    *h = c;
    return KL_OK;
}

int kl_destroy(kl_handle_t h) {
    if (!h) return KL_OK;
    Ctx *c = h;
    cudaSetDevice(c->device);
    // a borrowed stream (kl_set_stream) may already be destroyed by its owner -- e.g. another handle whose stream this
    // one was set to and which was destroyed first -- so it is not touched: wait for the device instead
    if (c->own_stream && c->stream) cudaStreamSynchronize(c->stream);
    else cudaDeviceSynchronize();
    for (int r = 0; r < 16; ++r)
        if (c->cb_peer[r] && c->cb_peer[r] != c->cb_local) cudaIpcCloseMemHandle(c->cb_peer[r]);
    cudaFree(c->cb_local);
    cudaFree(c->d_peerctl);
    if (c->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy((ncclComm_p)c->nccl_comm);
    cudaFree(c->d_S);
    cudaFree(c->d_I);
    cudaFree(c->d_partials);
    cudaFree(c->d_counter);
    cudaFree(c->d_hist);
    cudaFree(c->ws);
    cudaFree(c->d_halo);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->h_pinned_i) cudaFreeHost(c->h_pinned_i);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->ev3) cudaEventDestroy(c->ev3);
    prof_reset(c);
    graph_clear(c);
    if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
    for (auto e : c->prof_pool) cudaEventDestroy(e);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return KL_OK;
}

const char *kl_last_error(kl_handle_t h) { return h ? h->err.c_str() : "null handle"; }

int kl_set_stream(kl_handle_t h, void *cuda_stream) {
    if (!h) return KL_ERR_INVALID;
    Ctx *c = h;
    if (cuda_stream && !c->own_stream && c->stream == (cudaStream_t)cuda_stream) return KL_OK;
    cudaStreamSynchronize(c->stream);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    if (cuda_stream) {
        c->stream = (cudaStream_t)cuda_stream;
        c->own_stream = false;
    } else {
        KL_CUDA(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    return KL_OK;
}

int kl_get_stream(kl_handle_t h, void **cuda_stream) {
    if (!h || !cuda_stream) return KL_ERR_INVALID;
    *cuda_stream = (void *)h->stream;
    return KL_OK;
}

int kl_synchronize(kl_handle_t h) {
    if (!h) return KL_ERR_INVALID;
    KL_CUDA(h, cudaStreamSynchronize(h->stream));
    return KL_OK;
}

int kl_set_pointer_mode(kl_handle_t h, int mode) {
    if (!h || (mode != KL_POINTER_HOST && mode != KL_POINTER_DEVICE)) return KL_ERR_INVALID;
    h->pointer_mode = mode;
    return KL_OK;
}

int kl_set_option(kl_handle_t h, int key, int value) {
    if (!h) return KL_ERR_INVALID;
    switch (key) {
        case KL_OPT_ORTHO:
            if (value < KL_ORTHO_MGS2 || value > KL_ORTHO_CGS2_SELECTIVE) return KL_ERR_INVALID;
            h->opt_ortho = value;
            break;
        case KL_OPT_MAX_RESTARTS:
            if (value < 1) return KL_ERR_INVALID;
            h->opt_max_restarts = value;
            break;
        case KL_OPT_VERR: h->opt_verr = value != 0; break;
        case KL_OPT_CHECK_EVERY:
            if (value < 1) return KL_ERR_INVALID;
            h->opt_check_every = value;
            break;
        case KL_OPT_USE_GRAPH: h->opt_use_graph = value != 0; break;
        case KL_OPT_HH_MODE:
            if (value != KL_HH_SEQUENTIAL && value != KL_HH_BLOCKED) return KL_ERR_INVALID;
            h->opt_hh_mode = value;
            break;
        case KL_OPT_FUSE: h->opt_fuse = value != 0; break;
        case KL_OPT_PROFILE: h->opt_profile = value != 0; break;
        case KL_OPT_TMA: h->opt_tma = value != 0; break;
        case KL_OPT_CHAIN: h->opt_chain = value != 0; break;
        case KL_OPT_INLINE_ALLREDUCE: h->opt_inline_ar = value != 0; break;
        case KL_OPT_STENCIL_ROWS: h->opt_stencil_rows = value > 0 ? value : 0; break;
        case KL_OPT_REORTH_ETA:
            if (value < 1 || value > 1000) return KL_ERR_INVALID;
            h->opt_reorth_eta_permille = value;
            break;
        case KL_OPT_PEER:
            // all ranks must switch together; only meaningful before / between solves
            if (value && !h->peer_mapped) return KL_ERR_UNSUPPORTED;
            h->peer_ok = value != 0;
            break;
        case KL_OPT_PDL: h->opt_pdl = value != 0; break;
        case KL_OPT_STENCIL_TAIL: h->opt_stencil_tail = value; break;
        case KL_OPT_STENCIL_STAGGER: h->opt_stencil_stagger = value != 0; break;
        case KL_OPT_REVERSE: h->opt_reverse = value != 0; break;
        case KL_OPT_COOP: h->opt_coop = value != 0; break;
        case KL_OPT_PERSISTENT: h->opt_persistent = value != 0; break;
        case KL_OPT_PUSH_HALO: h->opt_push_halo = value != 0; break;
        case KL_OPT_CG_ONEPASS:
            if (value < -1 || value > 3) return KL_ERR_INVALID;
            h->opt_cg_onepass = value;
            break;
        case KL_OPT_X0:
            if (value != 0 && value != 1) return KL_ERR_INVALID;
            h->opt_x0 = value;
            break;
        default: return KL_ERR_INVALID;
    }
    return KL_OK;
}

int kl_get_option(kl_handle_t h, int key, int *value) {
    if (!h || !value) return KL_ERR_INVALID;
    switch (key) {
        case KL_OPT_ORTHO: *value = h->opt_ortho; break;
        case KL_OPT_MAX_RESTARTS: *value = h->opt_max_restarts; break;
        case KL_OPT_VERR: *value = h->opt_verr; break;
        case KL_OPT_CHECK_EVERY: *value = h->opt_check_every; break;
        case KL_OPT_USE_GRAPH: *value = h->opt_use_graph; break;
        case KL_OPT_HH_MODE: *value = h->opt_hh_mode; break;
        case KL_OPT_FUSE: *value = h->opt_fuse; break;
        case KL_OPT_PROFILE: *value = h->opt_profile; break;
        case KL_OPT_TMA: *value = h->opt_tma; break;
        case KL_OPT_CHAIN: *value = h->opt_chain; break;
        case KL_OPT_INLINE_ALLREDUCE: *value = h->opt_inline_ar; break;
        case KL_OPT_STENCIL_ROWS: *value = h->opt_stencil_rows; break;
        case KL_OPT_REORTH_ETA: *value = h->opt_reorth_eta_permille; break;
        case KL_OPT_PEER: *value = h->peer_ok ? 1 : 0; break;
        case KL_OPT_PDL: *value = h->opt_pdl; break;
        case KL_OPT_STENCIL_TAIL: *value = h->opt_stencil_tail; break;
        case KL_OPT_STENCIL_STAGGER: *value = h->opt_stencil_stagger; break;
        case KL_OPT_REVERSE: *value = h->opt_reverse; break;
        case KL_OPT_COOP: *value = h->opt_coop; break;
        case KL_OPT_PERSISTENT: *value = h->opt_persistent; break;
        case KL_OPT_PUSH_HALO: *value = h->opt_push_halo; break;
        case KL_OPT_CG_ONEPASS: *value = h->opt_cg_onepass; break;
        case KL_OPT_X0: *value = h->opt_x0; break;
        default: return KL_ERR_INVALID;
    }
    return KL_OK;
}

// ---- communicator -------------------------------------------------------
int kl_comm_unique_id(void *id_out) {
    if (!id_out) return KL_ERR_INVALID;
    static_assert(sizeof(ncclUniqueId_t) == KL_UNIQUE_ID_BYTES, "NCCL unique id size");
    std::string err;
    if (nccl_load(&err) != KL_OK) return KL_ERR_NCCL;
    ncclUniqueId_t id;
    if (g_nccl.GetUniqueId(&id) != 0) return KL_ERR_NCCL;
    memcpy(id_out, &id, sizeof id);
    return KL_OK;
}

int kl_comm_init(kl_handle_t h, int rank, int nranks, const void *id_bytes) {
    if (!h || nranks < 1 || rank < 0 || rank >= nranks) return KL_ERR_INVALID;
    Ctx *c = h;
    if (nranks == 1) {
        c->rank = 0;
        c->nranks = 1;
        return KL_OK;
    }
    if (!id_bytes) return KL_ERR_INVALID;
    if (nccl_load(&c->err) != KL_OK) return KL_ERR_NCCL;
    KL_CUDA(c, cudaSetDevice(c->device));
    ncclUniqueId_t id;
    memcpy(&id, id_bytes, sizeof id);
    ncclComm_p comm = nullptr;
    KL_NCCL(c, g_nccl.CommInitRank(&comm, nranks, id, rank));
    c->nccl_comm = comm;
    c->rank = rank;
    c->nranks = nranks;
    return peer_setup(c);
}

int kl_comm_rank(kl_handle_t h, int *rank, int *nranks) {
    if (!h) return KL_ERR_INVALID;
    if (rank) *rank = h->rank;
    if (nranks) *nranks = h->nranks;
    return KL_OK;
}

int kl_partition_rank(int ny, int rank, int nranks, int *j0, int *ny_local) {
    if (ny < 1 || nranks < 1 || rank < 0 || rank >= nranks) return KL_ERR_INVALID;
    // contiguous lines in memory order, the first (ny % P) ranks get one extra line
    const int base = ny / nranks, rem = ny % nranks;
    if (j0) *j0 = rank * base + (rank < rem ? rank : rem);
    if (ny_local) *ny_local = base + (rank < rem ? 1 : 0);
    return KL_OK;
}

int kl_partition(kl_handle_t h, int ny, int *j0, int *ny_local) {
    if (!h) return KL_ERR_INVALID;
    return kl_partition_rank(ny, h->rank, h->nranks, j0, ny_local);
}

// ---- device vectors -------------------------------------------------------
int kl_vec_alloc(kl_handle_t h, size_t n, double **d_ptr) {
    if (!h || !d_ptr) return KL_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaError_t e = cudaMalloc((void **)d_ptr, n * sizeof(double));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return h->fail(KL_ERR_ALLOC, "kl_vec_alloc", e);
    }
    return KL_OK;
}
int kl_vec_free(kl_handle_t h, double *d_ptr) {
    if (!h) return KL_ERR_INVALID;
    cudaStreamSynchronize(h->stream);
    KL_CUDA(h, cudaFree(d_ptr));
    return KL_OK;
}
int kl_vec_upload(kl_handle_t h, double *d_dst, const double *h_src, size_t n) {
    if (!h) return KL_ERR_INVALID;
    KL_CUDA(h, cudaMemcpyAsync(d_dst, h_src, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    KL_CUDA(h, cudaStreamSynchronize(h->stream));
    return KL_OK;
}
int kl_vec_download(kl_handle_t h, double *h_dst, const double *d_src, size_t n) {
    if (!h) return KL_ERR_INVALID;
    KL_CUDA(h, cudaMemcpyAsync(h_dst, d_src, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    KL_CUDA(h, cudaStreamSynchronize(h->stream));
    return KL_OK;
}

int kl_get_history(kl_handle_t h, double *out, int cap, int *len) {
    if (!h) return KL_ERR_INVALID;
    if (len) *len = h->history_len;
    if (out && cap > 0) {
        int k = h->history_len < cap ? h->history_len : cap;
        if (k > (int)h->history.size()) k = (int)h->history.size();
        memcpy(out, h->history.data(), sizeof(double) * k);
    }
    return KL_OK;
}

int kl_get_stats(kl_handle_t h, kl_stats_t *out) {
    if (!h || !out) return KL_ERR_INVALID;
    *out = h->stats;
    return KL_OK;
}

int kl_get_profile(kl_handle_t h, int idx, const char **name, double *ms, long long *launches,
                   double *algorithmic_bytes) {
    if (!h || idx < 0 || idx >= KL_PROFILE_CLASSES) return KL_ERR_INVALID;
    if (name) *name = h->prof_name[idx];
    if (ms) *ms = h->prof_ms[idx];
    if (launches) *launches = h->prof_launches[idx];
    if (algorithmic_bytes) *algorithmic_bytes = h->prof_bytes[idx];
    return KL_OK;
}

int kl_cheb_params_from_ritz(double theta_min, double theta_max, double params_out[2]) {
    (void)theta_min;
    if (!params_out || !(theta_max > 0)) return KL_ERR_INVALID;
    // tests/test_poisson_mf.f90:38 passes (8.2, 0.2) for a spectrum whose top is 8:
    // (1.025 lambda_max, 1.025 lambda_max / 41), "max first".
    params_out[0] = 1.025 * theta_max;
    params_out[1] = params_out[0] / 41.0;
    return KL_OK;
}

// Interval for the degree-k Chebyshev preconditioner (KL_PC_CHEB) from a Lanczos estimate: [b/ratio, b] with
// b = 1.025 theta_max and a ratio that grows with the degree -- a degree-k polynomial can cover a wider part of
// the spectrum.  The ratios are the best ones of the sweep in profiles/r01_cheb_sweep_2048.json (GMRES(95) and PCG
// on the 2048^2 Poisson grid): 41 (the reference's cbpr2 policy) for k = 1, 100 for k = 2, 400 for k = 3..4,
// 1000 above.  Host arithmetic only.
int kl_cheb_interval_from_ritz(double theta_max, int degree, double params_out[2]) {
    if (!params_out || !(theta_max > 0) || degree < 1) return KL_ERR_INVALID;
    const double ratio = degree <= 1 ? 41.0 : (degree == 2 ? 100.0 : (degree <= 4 ? 400.0 : 1000.0));
    params_out[0] = 1.025 * theta_max;
    params_out[1] = params_out[0] / ratio;
    return KL_OK;
}

}  // extern "C"
