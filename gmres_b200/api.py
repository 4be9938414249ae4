"""ctypes binding of include/krylov_b200.h and the Python mirror of the reference API.

Every solver method keeps the reference procedure's name and argument order
(citations are to the reference tree):

    gmres_mgsr_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,restart_out,M_inv,params)  src/gmres_mgsr.f90:277
    gmres_mgsr_mf (...)                                                              src/gmres_mgsr.f90:98
    gmres_hh_omp(Ax_vec,b,x,m,tol,final_err,v_err,n_out,stages_out)                  src/gmres_hh.f90:211
    gmres_hh_prec_omp(...,m_inv,params)                                              src/gmres_hh.f90:388
    cg / cg_omp (Ax_op,b,x,tol,iter,res)                                             src/cg.f90:11 / :83
    pcg / pcg_omp (...,M_inv,params)                                                 src/cg.f90:44 / :154
    bicgstab / pbicgstab / pbicgstab_omp                                             src/bicgstab.f90:12 / :49 / :91

intent(out) arguments become fields of the returned result object.  Vectors may be
numpy float64 arrays (host pointer mode; copied to and from the device inside the
call) or CUDA torch.float64 tensors (device pointer mode; they stay in HBM).

Every solver method also takes `x0=None`: an initial guess of b's kind and length
(KL_OPT_X0).  The reference starts from x = 0, and so does a call without x0.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBNAME = "libkrylov_b200.so"

KL_OK, KL_NOT_CONVERGED, KL_BREAKDOWN = 0, 1, 2
KL_OP_POISSON5, KL_OP_POISSON5_BRANCHY, KL_OP_ANISO5, KL_OP_ANISO5_VAR, KL_OP_STENCIL5, KL_OP_USER = 0, 1, 2, 4, 5, 100
KL_ERR_INVALID, KL_ERR_UNSUPPORTED = -1, -5
KL_PC_NONE, KL_PC_CBPR2, KL_PC_CHEB, KL_PC_JACOBI_CHEB, KL_PC_USER = 0, 1, 2, 3, 100
KL_POINTER_HOST, KL_POINTER_DEVICE = 0, 1
(KL_OPT_ORTHO, KL_OPT_MAX_RESTARTS, KL_OPT_VERR, KL_OPT_CHECK_EVERY, KL_OPT_USE_GRAPH,
 KL_OPT_HH_MODE, KL_OPT_FUSE, KL_OPT_PROFILE) = range(1, 9)
KL_OPT_TMA, KL_OPT_PEER, KL_OPT_REORTH_ETA, KL_OPT_CHAIN, KL_OPT_STENCIL_ROWS, KL_OPT_INLINE_ALLREDUCE = 9, 10, 11, 12, 13, 14
KL_OPT_X0 = 23
ORTHO_MGS2, ORTHO_CGS2, ORTHO_CGS2_SELECTIVE = 0, 1, 2
HH_SEQUENTIAL, HH_BLOCKED = 0, 1
KL_UNIQUE_ID_BYTES = 128

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

APPLY_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p)
PRECOND_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                         C.c_void_p, _dp, C.c_int, C.c_int, C.c_int, C.c_void_p)


class kl_operator_t(C.Structure):
    _fields_ = [("kind", C.c_int), ("eps_x", C.c_double), ("eps_y", C.c_double),
                ("fn", APPLY_FN), ("user", C.c_void_p)]


class kl_aniso_var_t(C.Structure):
    _fields_ = [("kx", C.c_void_p), ("ky", C.c_void_p)]


class kl_stencil5_t(C.Structure):
    _fields_ = [("c", C.c_double), ("wl", C.c_double), ("wr", C.c_double), ("wd", C.c_double), ("wu", C.c_double)]


class kl_precond_t(C.Structure):
    _fields_ = [("kind", C.c_int), ("degree", C.c_int), ("fn", PRECOND_FN), ("user", C.c_void_p)]


class kl_stats_t(C.Structure):
    _fields_ = [("iterations", C.c_int), ("cycles", C.c_int), ("solve_ms", C.c_double),
                ("total_ms", C.c_double), ("algorithmic_bytes", C.c_double),
                ("kernel_launches", C.c_longlong), ("orth_frobenius", C.c_double),
                ("h2d_bytes", C.c_double), ("d2h_bytes", C.c_double), ("reorth_skipped", C.c_int)]


class KrylovError(RuntimeError):
    pass


def library_path() -> str:
    return os.environ.get("KRYLOV_B200_LIB", os.path.join(_HERE, _LIBNAME))


_lib = None


def load_library():
    """Load libkrylov_b200.so.  Raises (never falls back to a CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise KrylovError(
            f"{path} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; "
            "g.build()' or make -C gmres_b200/csrc).  There is no CPU fallback.")
    L = C.CDLL(path)
    L.kl_last_error.restype = C.c_char_p
    L.kl_last_error.argtypes = [C.c_void_p]
    for name in ("kl_create",):
        getattr(L, name).argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.kl_destroy.argtypes = [C.c_void_p]
    L.kl_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.kl_get_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.kl_synchronize.argtypes = [C.c_void_p]
    L.kl_set_pointer_mode.argtypes = [C.c_void_p, C.c_int]
    L.kl_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.kl_get_option.argtypes = [C.c_void_p, C.c_int, _ip]
    L.kl_comm_unique_id.argtypes = [C.c_void_p]
    L.kl_comm_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.kl_comm_rank.argtypes = [C.c_void_p, _ip, _ip]
    L.kl_partition.argtypes = [C.c_void_p, C.c_int, _ip, _ip]
    L.kl_apply_operator.argtypes = [C.c_void_p, C.POINTER(kl_operator_t), C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int]
    L.kl_apply_precond.argtypes = [C.c_void_p, C.POINTER(kl_precond_t), C.POINTER(kl_operator_t),
                                   C.c_void_p, C.c_void_p, _dp, C.c_int, C.c_int, C.c_int]
    gm = [C.c_void_p, C.POINTER(kl_operator_t), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
          C.c_double, _dp, _dp, _ip, _ip]
    pc = [C.POINTER(kl_precond_t), _dp, C.c_int]
    L.kl_gmres_mgsr_omp.argtypes = gm + pc
    L.kl_gmres_mgsr_mf.argtypes = gm + pc
    L.kl_gmres_hh_omp.argtypes = gm
    L.kl_gmres_hh_prec_omp.argtypes = gm + pc
    cg = [C.c_void_p, C.POINTER(kl_operator_t), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double,
          _ip, _dp]
    for name in ("kl_cg", "kl_cg_omp", "kl_bicgstab"):
        getattr(L, name).argtypes = cg
    for name in ("kl_pcg", "kl_pcg_omp", "kl_pbicgstab", "kl_pbicgstab_omp"):
        getattr(L, name).argtypes = cg + pc
    dn = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, _dp, _dp, _ip, _ip]
    L.kl_gmres_mgsr_dense.argtypes = dn
    L.kl_gmres_hh_dense.argtypes = dn
    L.kl_generate_matrix.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.kl_dense_matvec.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.kl_lanczos.argtypes = [C.c_void_p, C.POINTER(kl_operator_t), C.c_int, C.c_int, C.c_int, _dp, _dp]
    L.kl_cheb_params_from_ritz.argtypes = [C.c_double, C.c_double, _dp]
    L.kl_cheb_interval_from_ritz.argtypes = [C.c_double, C.c_int, _dp]
    L.kl_stencil5_spectrum.argtypes = [C.POINTER(kl_stencil5_t), C.c_int, C.c_int, _dp, _dp]
    L.kl_get_history.argtypes = [C.c_void_p, _dp, C.c_int, _ip]
    L.kl_get_stats.argtypes = [C.c_void_p, C.POINTER(kl_stats_t)]
    L.kl_get_profile.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), _dp, C.POINTER(C.c_longlong), _dp]
    L.kl_vec_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.kl_vec_free.argtypes = [C.c_void_p, C.c_void_p]
    L.kl_vec_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.kl_vec_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    _lib = L
    return L


# --------------------------------------------------------------------------
# plug-ins: the reference passes procedures; here they are descriptors
# --------------------------------------------------------------------------
@dataclass(frozen=True)
class Operator:
    """procedure(stencil_vector) -- src/interfaces.f90:12-18."""
    kind: int
    eps_x: float = 1.0
    eps_y: float = 1.0
    fn: Optional[object] = None  # python callable(d_x:int, d_y:int, nx, ny_local, stream:int) for KL_OP_USER
    coef: Optional[tuple] = None  # (kx, ky) CUDA float64 tensors for KL_OP_ANISO5_VAR
    w5: Optional[tuple] = None    # (c, wl, wr, wd, wu) for KL_OP_STENCIL5

    def _c(self):
        o = kl_operator_t()
        o.kind, o.eps_x, o.eps_y = self.kind, self.eps_x, self.eps_y
        keep = None
        if self.kind == KL_OP_ANISO5_VAR:
            kx, ky = self.coef
            keep = kl_aniso_var_t(C.c_void_p(kx.data_ptr()), C.c_void_p(ky.data_ptr()))
            o.user = C.cast(C.pointer(keep), C.c_void_p)
        if self.kind == KL_OP_STENCIL5:
            keep = kl_stencil5_t(*self.w5)
            o.user = C.cast(C.pointer(keep), C.c_void_p)
        if self.kind == KL_OP_USER:
            f = self.fn

            def tramp(user, dx, dy, nx, nyl, stream):
                try:
                    f(dx, dy, nx, nyl, stream)
                    return 0
                except Exception:  # pragma: no cover
                    import traceback
                    traceback.print_exc()
                    return 1

            keep = APPLY_FN(tramp)
            o.fn = keep
        return o, keep


@dataclass(frozen=True)
class Precond:
    """procedure(precond) -- src/interfaces.f90:19-28.

    KL_PC_USER: `fn(A_x, d_r, d_z, d_aux, params, nx, ny_local, stream)` mirrors the reference's
    `subroutine precond(A_x, r, z, aux, params, n)`: A_x is the solver's operator (an opaque
    `const kl_operator_t *` that can be handed to kl_apply_operator), d_r / d_z / d_aux are device pointers
    (aux is the solver's scratch vector, lent to the preconditioner as in gmres_mgsr.f90:302,337), params the
    solver's params array.  Enqueue-only on `stream`; it must not synchronise."""
    kind: int
    degree: int = 0
    fn: Optional[object] = None

    def _c(self):
        p = kl_precond_t()
        p.kind, p.degree = self.kind, self.degree
        keep = None
        if self.kind == KL_PC_USER:
            f = self.fn
            if f is None:
                raise KrylovError("Precond(KL_PC_USER) needs fn")

            def tramp(h, a_x, user, d_r, d_z, d_aux, params, nparams, nx, nyl, stream):
                try:
                    f(a_x, d_r, d_z, d_aux, [params[i] for i in range(nparams)], nx, nyl, stream)
                    return 0
                except Exception:  # pragma: no cover
                    import traceback
                    traceback.print_exc()
                    return 1

            keep = PRECOND_FN(tramp)
            p.fn = keep
        return p, keep


stvec = Operator(KL_OP_POISSON5)                 # poisson::stvec        src/problems/poisson.f90:33
stv_poisson = Operator(KL_OP_POISSON5_BRANCHY)   # poisson::stv_poisson  src/problems/poisson.f90:79
cbpr2 = Precond(KL_PC_CBPR2)                     # chebyshev_precond::cbpr2  src/preconds/chebyshev.f90:8
no_precond = Precond(KL_PC_NONE)


def aniso(eps_x: float, eps_y: float) -> Operator:
    return Operator(KL_OP_ANISO5, float(eps_x), float(eps_y))


def aniso_var(kx, ky) -> Operator:
    """Variable-coefficient anisotropic diffusion (KL_OP_ANISO5_VAR): cell coefficient grids kx(i,j), ky(i,j) as numpy
    arrays or CUDA tensors of nx*ny values (idx = i + j*nx); they are kept on the device by the returned descriptor."""
    import torch

    def dev(a):
        if _is_torch_cuda(a):
            return a.contiguous().reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(-1)).cuda()

    return Operator(KL_OP_ANISO5_VAR, coef=(dev(kx), dev(ky)))


def stencil5(c: float, wl: float, wr: float, wd: float, wu: float) -> Operator:
    """General constant-coefficient 5-point operator with zero Dirichlet boundary (KL_OP_STENCIL5):
        y(i,j) = c x(i,j) - (wl x(i-1,j) + wr x(i+1,j) + wd x(i,j+1) + wu x(i,j-1)),   idx = i + j*nx
    ("d" is the next line idx+nx, "u" the previous one idx-nx).  Every weight must be a finite real number.  It is
    nonsymmetric unless wl == wr and wd == wu; CG, PCG and lanczos refuse it then.  One GPU only."""
    w = []
    for name, v in (("c", c), ("wl", wl), ("wr", wr), ("wd", wd), ("wu", wu)):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)):
            raise KrylovError(f"stencil5: weight {name} must be a real number, got {type(v).__name__}")
        f = float(v)
        if not np.isfinite(f):
            raise KrylovError(f"stencil5: weight {name} must be finite, got {f}")
        w.append(f)
    return Operator(KL_OP_STENCIL5, w5=tuple(w))


def convdiff(px: float, py: float, upwind: bool = False) -> Operator:
    """Convection-diffusion -lap(u) + b.grad(u) on a grid of spacing h, scaled by h^2 (KL_OP_STENCIL5), in terms of the
    cell Peclet numbers px = bx*h/2 and py = by*h/2.
      central: c = 4, wl = 1 + px, wr = 1 - px, wu = 1 + py, wd = 1 - py.  The spectrum is real iff |px|, |py| <= 1.
      upwind (first order): c = (4 + 2|px|) + 2|py|; the upstream weight (wl for px > 0, wr for px < 0; wu for py > 0,
      wd for py < 0) is 1 + 2|p|, the other one 1.  The spectrum is always real."""
    for name, v in (("px", px), ("py", py)):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)) or \
                not np.isfinite(float(v)):
            raise KrylovError(f"convdiff: {name} must be a finite real number")
    px, py = float(px), float(py)
    if not upwind:
        return stencil5(4.0, 1.0 + px, 1.0 - px, 1.0 - py, 1.0 + py)
    ax, ay = abs(px), abs(py)
    wl, wr = (1.0 + 2.0 * ax, 1.0) if px >= 0 else (1.0, 1.0 + 2.0 * ax)
    wu, wd = (1.0 + 2.0 * ay, 1.0) if py >= 0 else (1.0, 1.0 + 2.0 * ay)
    return stencil5((4.0 + 2.0 * ax) + 2.0 * ay, wl, wr, wd, wu)


def stencil5_spectrum(op: Operator, nx: int, ny: int):
    """(lam_min, lam_max): the exact extremes of the Dirichlet spectrum of a stencil5 operator on an nx x ny grid
    (kl_stencil5_spectrum, host arithmetic, no GPU needed).  Raises KrylovError when the spectrum is complex
    (wl*wr < 0 or wd*wu < 0).  (lam_min, lam_max) is the exact interval for cheb(k)."""
    if not isinstance(op, Operator) or op.kind != KL_OP_STENCIL5:
        raise KrylovError("stencil5_spectrum: op must be a stencil5 / convdiff operator")
    if int(nx) < 1 or int(ny) < 1:
        raise KrylovError("stencil5_spectrum: nx, ny >= 1")
    w = kl_stencil5_t(*op.w5)
    lo, hi = C.c_double(), C.c_double()
    rc = load_library().kl_stencil5_spectrum(C.byref(w), int(nx), int(ny), C.byref(lo), C.byref(hi))
    if rc == KL_ERR_UNSUPPORTED:
        raise KrylovError("stencil5_spectrum: the spectrum is complex (wl*wr < 0 or wd*wu < 0)")
    if rc != 0:
        raise KrylovError(f"kl_stencil5_spectrum failed with {rc}")
    return lo.value, hi.value


def cheb(degree: int) -> Precond:
    return Precond(KL_PC_CHEB, int(degree))


def jacobi_cheb(degree: int) -> Precond:
    """Chebyshev of the given degree on the Jacobi-scaled operator D^-1 A (KL_PC_JACOBI_CHEB), for aniso_var operators.
    Degree 0 is point Jacobi (params ignored); degree k >= 1 takes params = (a, b), an interval of the spectrum of
    D^-1 A, which lies in (0, 2]."""
    return Precond(KL_PC_JACOBI_CHEB, int(degree))


@dataclass
class GmresResult:
    x: object
    final_err: np.ndarray
    v_err: np.ndarray
    n_out: int
    restart_out: int          # restart_out / stages_out
    status: int
    history: np.ndarray = field(default_factory=lambda: np.zeros(0))
    stats: dict = field(default_factory=dict)


@dataclass
class CgResult:
    x: object
    iter: int
    res: float
    status: int
    history: np.ndarray = field(default_factory=lambda: np.zeros(0))
    stats: dict = field(default_factory=dict)


def _is_torch_cuda(a) -> bool:
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda") and a.is_cuda


class Handle:
    """kl_handle_t: one per GPU (one process per GPU for multi-GPU runs)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._L = load_library()
        self._h = C.c_void_p()
        rc = self._L.kl_create(C.byref(self._h), int(device))
        if rc != 0:
            raise KrylovError(f"kl_create(device={device}) failed with {rc}: no usable CUDA device "
                              "(this library has no CPU path)")
        self.device = int(device)
        self.rank, self.nranks = 0, 1
        self._user_stream = stream is not None
        self._bound_stream = None                  # (pointer, torch ExternalStream) of the handle's stream
        if stream is not None:
            self._chk(self._L.kl_set_stream(self._h, C.c_void_p(stream)))

    # -- plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._L.kl_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc, allow=(0,)):
        if rc not in allow:
            msg = self._L.kl_last_error(self._h)
            raise KrylovError(f"libkrylov_b200 error {rc}: {msg.decode() if msg else ''}")
        return rc

    def set_option(self, key: int, value: int):
        self._chk(self._L.kl_set_option(self._h, key, int(value)))

    def get_option(self, key: int) -> int:
        v = C.c_int()
        self._chk(self._L.kl_get_option(self._h, key, C.byref(v)))
        return v.value

    def set_ortho(self, mode: int):
        self.set_option(KL_OPT_ORTHO, mode)

    def set_stream(self, stream: Optional[int]):
        """Run on an existing CUDA stream (None: the handle's own stream).  Device-pointer calls are ordered against
        torch's current stream with events either way (_order_in / _order_out)."""
        self._chk(self._L.kl_set_stream(self._h, C.c_void_p(stream or 0)))
        self._user_stream = stream is not None
        self._bound_stream = None

    def _lib_stream(self):
        """the handle's stream as a torch.cuda.ExternalStream (for event-based ordering)"""
        import torch
        p = C.c_void_p()
        self._chk(self._L.kl_get_stream(self._h, C.byref(p)))
        if self._bound_stream is None or self._bound_stream[0] != (p.value or 0):
            self._bound_stream = (p.value or 0, torch.cuda.ExternalStream(p.value or 0, device=torch.device("cuda", self.device)))
        return self._bound_stream[1]

    def _order_in(self):
        """Device-pointer mode: the library's stream (cudaStreamNonBlocking, it does not synchronise with torch's
        streams by itself) waits for everything already enqueued on torch's CURRENT stream -- the producers of the
        input tensors.  Kernels still run on the handle's own stream (running them on torch's legacy default
        stream cost the fused CG kernels their programmatic-dependent-launch overlap)."""
        import torch
        self._lib_stream().wait_stream(torch.cuda.current_stream(self.device))

    def _order_out(self):
        """... and torch's current stream waits for the library's work, so that consumers of the outputs (and the
        caching allocator, when an input tensor is freed right after the call) are ordered after it."""
        import torch
        torch.cuda.current_stream(self.device).wait_stream(self._lib_stream())

    def synchronize(self):
        self._chk(self._L.kl_synchronize(self._h))

    def comm_init(self, rank: int, nranks: int, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), KL_UNIQUE_ID_BYTES)
        self._chk(self._L.kl_comm_init(self._h, rank, nranks, buf))
        self.rank, self.nranks = rank, nranks

    def unique_id(self) -> bytes:
        buf = C.create_string_buffer(KL_UNIQUE_ID_BYTES)
        rc = self._L.kl_comm_unique_id(buf)
        if rc != 0:
            raise KrylovError(f"kl_comm_unique_id failed: {rc}")
        return buf.raw

    def partition(self, ny: int):
        j0, nyl = C.c_int(), C.c_int()
        self._chk(self._L.kl_partition(self._h, ny, C.byref(j0), C.byref(nyl)))
        return j0.value, nyl.value

    def stats(self) -> dict:
        s = kl_stats_t()
        self._chk(self._L.kl_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in s._fields_}

    def profile(self) -> list:
        """Per-kernel-class CUDA-event timers of the last solve (KL_OPT_PROFILE = 1)."""
        out = []
        for i in range(8):
            name, ms, ln, by = C.c_char_p(), C.c_double(), C.c_longlong(), C.c_double()
            if self._L.kl_get_profile(self._h, i, C.byref(name), C.byref(ms), C.byref(ln), C.byref(by)) != 0:
                break
            if ln.value:
                out.append(dict(name=name.value.decode() if name.value else f"class{i}", ms=ms.value,
                                launches=ln.value, algorithmic_bytes=by.value))
        return out

    def history(self) -> np.ndarray:
        n = C.c_int()
        self._L.kl_get_history(self._h, None, 0, C.byref(n))
        out = np.zeros(max(n.value, 1))
        self._L.kl_get_history(self._h, out.ctypes.data_as(_dp), out.size, C.byref(n))
        return out[: n.value]

    # -- vector marshalling
    def _in(self, a, n_expected=None):
        if _is_torch_cuda(a):
            import torch
            assert a.dtype == torch.float64 and a.is_contiguous()
            self._chk(self._L.kl_set_pointer_mode(self._h, KL_POINTER_DEVICE))
            self._order_in()
            return a, C.c_void_p(a.data_ptr()), True
        arr = np.ascontiguousarray(a, dtype=np.float64)
        self._chk(self._L.kl_set_pointer_mode(self._h, KL_POINTER_HOST))
        return arr, C.c_void_p(arr.ctypes.data), False

    def set_output_buffer(self, buf):
        """Use `buf` (numpy array, e.g. a view of pinned memory, or CUDA tensor) for the next
        solver call's x instead of allocating one (the reference's x is allocatable,intent(out))."""
        self._xbuf = buf

    def _out_like(self, a, is_dev):
        buf = getattr(self, "_xbuf", None)
        if buf is not None:
            self._xbuf = None
            if is_dev:
                return buf, C.c_void_p(buf.data_ptr())
            return buf, C.c_void_p(buf.ctypes.data)
        if is_dev:
            import torch
            o = torch.empty_like(a)
            return o, C.c_void_p(o.data_ptr())
        o = np.empty_like(a)
        return o, C.c_void_p(o.ctypes.data)

    @staticmethod
    def _check_x0(x0, b):
        """x0 must be b's kind (a CUDA float64 tensor on b's device, or a numpy array) and length; checked before any
        call into the library."""
        if x0 is None:
            return
        if _is_torch_cuda(b):
            import torch
            if not (_is_torch_cuda(x0) and x0.dtype == torch.float64 and x0.device == b.device):
                raise KrylovError("x0 must be a CUDA float64 tensor on b's device when b is one")
            nb, n0 = b.numel(), x0.numel()
        else:
            if not isinstance(x0, np.ndarray):
                raise KrylovError("x0 must be a numpy array when b is not a CUDA tensor")
            nb, n0 = np.asarray(b).size, x0.size
        if n0 != nb:
            raise KrylovError(f"x0 has {n0} values, b has {nb}")

    def _x_out(self, ba, dev, x0):
        """The solver's x buffer (see _out_like).  KL_OPT_X0 is set on every call, so that a value left on the handle
        can never make a call read an uninitialised buffer; with x0 given, x0 is copied into the buffer (the caller's
        x0 is not written) and the library starts from it."""
        self._chk(self._L.kl_set_option(self._h, KL_OPT_X0, 0 if x0 is None else 1))
        x, xp = self._out_like(ba, dev)
        if x0 is not None:
            if dev:
                x.view(-1).copy_(x0.reshape(-1))
                self._order_in()     # the library's stream waits for the copy on torch's current stream
            else:
                x.reshape(-1)[:] = x0.reshape(-1)
        return x, xp

    @staticmethod
    def _grid(b, nx, ny):
        n = b.numel() if hasattr(b, "numel") else b.size
        if nx is None:
            # nsize = int(sqrt(real(n)))  (gmres_mgsr.f90:298) -- single precision sqrt
            nx = ny = int(np.sqrt(np.float32(n)))
        return int(nx), int(ny)

    # -- operator / preconditioner application
    def apply(self, A: Operator, x, nx: int, ny: int):
        """call stvec(x, y, n)  (src/problems/poisson.f90:33)."""
        xa, xp, dev = self._in(x)
        y, yp = self._out_like(xa, dev)
        o, keep = A._c()
        self._chk(self._L.kl_apply_operator(self._h, C.byref(o), xp, yp, nx, ny))
        if dev:
            self._order_out()
        return y

    def apply_precond(self, M: Precond, A: Operator, r, params: Sequence[float], nx: int, ny: int):
        """call cbpr2(A_x, r, z, aux, params, n)  (src/preconds/chebyshev.f90:8)."""
        ra, rp, dev = self._in(r)
        z, zp = self._out_like(ra, dev)
        o, keep = A._c()
        p, keep_p = M._c()
        pr = np.ascontiguousarray(params, dtype=np.float64)
        self._chk(self._L.kl_apply_precond(self._h, C.byref(p), C.byref(o), rp, zp,
                                           pr.ctypes.data_as(_dp), pr.size, nx, ny))
        if dev:
            self._order_out()
        return z

    # -- GMRES
    def _gmres(self, fn, A, b, m, tol, M, params, nx, ny, with_pc=True, x0=None):
        self._check_x0(x0, b)
        ba, bp, dev = self._in(b)
        nx, ny = self._grid(ba, nx, ny)
        x, xp = self._x_out(ba, dev, x0)
        fe = np.zeros(m)
        ve = np.zeros(m + 1)
        n_out, rs = C.c_int(0), C.c_int(0)
        o, keep = A._c()
        args = [self._h, C.byref(o), bp, xp, nx, ny, int(m), float(tol), fe.ctypes.data_as(_dp),
                ve.ctypes.data_as(_dp), C.byref(n_out), C.byref(rs)]
        if with_pc:
            p, keep_p = (M or no_precond)._c()
            pr = np.ascontiguousarray(params if params is not None else (0.0, 0.0), dtype=np.float64)
            args += [C.byref(p), pr.ctypes.data_as(_dp), pr.size]
        rc = self._chk(fn(*args), allow=(KL_OK, KL_NOT_CONVERGED, KL_BREAKDOWN))
        if dev:
            self._order_out()
        return GmresResult(x, fe, ve, n_out.value, rs.value, rc, self.history(), self.stats())

    def gmres_mgsr_omp(self, Ax_vec, b, m, tol, M_inv=None, params=None, nx=None, ny=None, x0=None):
        return self._gmres(self._L.kl_gmres_mgsr_omp, Ax_vec, b, m, tol, M_inv, params, nx, ny, x0=x0)

    def gmres_mgsr_mf(self, Ax_vec, b, m, tol, M_inv=None, params=None, nx=None, ny=None, x0=None):
        return self._gmres(self._L.kl_gmres_mgsr_mf, Ax_vec, b, m, tol, M_inv, params, nx, ny, x0=x0)

    def gmres_hh_omp(self, Ax_vec, b, m, tol, nx=None, ny=None, x0=None):
        return self._gmres(self._L.kl_gmres_hh_omp, Ax_vec, b, m, tol, None, None, nx, ny, with_pc=False, x0=x0)

    def gmres_hh_prec_omp(self, Ax_vec, b, m, tol, m_inv=None, params=None, nx=None, ny=None, x0=None):
        return self._gmres(self._L.kl_gmres_hh_prec_omp, Ax_vec, b, m, tol, m_inv, params, nx, ny, x0=x0)

    # -- dense-operator variants (src/gmres_mgsr.f90:11, src/gmres_hh.f90:10, src/problems/hilbert.f90:6)
    def _dense_in(self, A, n):
        """A(n,n) as the Fortran array.  numpy: any layout (copied to column-major); CUDA tensor: its memory
        must already be column-major (pass A.t().contiguous() of a row-major torch matrix)."""
        if _is_torch_cuda(A):
            assert A.numel() == n * n and A.is_contiguous()
            return A, C.c_void_p(A.data_ptr())
        Af = np.asfortranarray(A, dtype=np.float64)
        assert Af.shape == (n, n)
        return Af, C.c_void_p(Af.ctypes.data)

    def generate_matrix(self, n: int) -> np.ndarray:
        """call generate_matrix(H, n)  (hilbert::generate_matrix, src/problems/hilbert.f90:6)."""
        self._chk(self._L.kl_set_pointer_mode(self._h, KL_POINTER_HOST))
        H = np.zeros((n, n), order="F")
        self._chk(self._L.kl_generate_matrix(self._h, C.c_void_p(H.ctypes.data), int(n)))
        return H

    def dense_matvec(self, A, x):
        """y = matmul(A, x)  (tests/test_hilbert.f90:44-45 builds b this way)."""
        xa, xp, dev = self._in(x)
        n = xa.numel() if dev else xa.size
        Aa, Ap = self._dense_in(A, n)
        y, yp = self._out_like(xa, dev)
        self._chk(self._L.kl_dense_matvec(self._h, Ap, n, xp, yp))
        if dev:
            self._order_out()
        return y

    def _gmres_dense(self, fn, A, b, m, tol, x0=None):
        self._check_x0(x0, b)
        ba, bp, dev = self._in(b)
        n = ba.numel() if dev else ba.size
        Aa, Ap = self._dense_in(A, n)
        x, xp = self._x_out(ba, dev, x0)
        fe = np.zeros(m)
        ve = np.zeros(m + 1)
        n_out, rs = C.c_int(0), C.c_int(0)
        rc = self._chk(fn(self._h, Ap, n, bp, xp, int(m), float(tol), fe.ctypes.data_as(_dp),
                          ve.ctypes.data_as(_dp), C.byref(n_out), C.byref(rs)),
                       allow=(KL_OK, KL_NOT_CONVERGED, KL_BREAKDOWN))
        if dev:
            self._order_out()
        return GmresResult(x, fe, ve, n_out.value, rs.value, rc, self.history(), self.stats())

    def gmres_mgsr_dense(self, A, b, m, tol, x0=None):
        return self._gmres_dense(self._L.kl_gmres_mgsr_dense, A, b, m, tol, x0)

    def gmres_hh_dense(self, A, b, m, tol, x0=None):
        return self._gmres_dense(self._L.kl_gmres_hh_dense, A, b, m, tol, x0)

    # -- CG / BiCGSTAB
    def _cg(self, fn, A, b, tol, it, M, params, nx, ny, with_pc, x0=None):
        self._check_x0(x0, b)
        ba, bp, dev = self._in(b)
        nx, ny = self._grid(ba, nx, ny)
        x, xp = self._x_out(ba, dev, x0)
        itc, res = C.c_int(int(it)), C.c_double(0.0)
        o, keep = A._c()
        args = [self._h, C.byref(o), bp, xp, nx, ny, float(tol), C.byref(itc), C.byref(res)]
        if with_pc:
            p, keep_p = (M or no_precond)._c()
            pr = np.ascontiguousarray(params if params is not None else (0.0, 0.0), dtype=np.float64)
            args += [C.byref(p), pr.ctypes.data_as(_dp), pr.size]
        rc = self._chk(fn(*args), allow=(KL_OK, KL_NOT_CONVERGED, KL_BREAKDOWN))
        if dev:
            self._order_out()
        return CgResult(x, itc.value, res.value, rc, self.history(), self.stats())

    def cg(self, Ax_op, b, tol, iter, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_cg, Ax_op, b, tol, iter, None, None, nx, ny, False, x0)

    def cg_omp(self, Ax_op, b, tol, iter, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_cg_omp, Ax_op, b, tol, iter, None, None, nx, ny, False, x0)

    def pcg(self, Ax_op, b, tol, iter, M_inv, params, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_pcg, Ax_op, b, tol, iter, M_inv, params, nx, ny, True, x0)

    def pcg_omp(self, Ax_op, b, tol, iter, M_inv, params, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_pcg_omp, Ax_op, b, tol, iter, M_inv, params, nx, ny, True, x0)

    def bicgstab(self, ax_op, b, tol, iter, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_bicgstab, ax_op, b, tol, iter, None, None, nx, ny, False, x0)

    def pbicgstab(self, ax_op, b, tol, iter, m_inv, params, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_pbicgstab, ax_op, b, tol, iter, m_inv, params, nx, ny, True, x0)

    def pbicgstab_omp(self, ax_op, b, tol, max_iter, m_inv, params, nx=None, ny=None, x0=None):
        return self._cg(self._L.kl_pbicgstab_omp, ax_op, b, tol, max_iter, m_inv, params, nx, ny, True, x0)

    # -- Lanczos
    def lanczos(self, A: Operator, nx: int, ny: int, steps: int = 30):
        lo, hi = C.c_double(), C.c_double()
        o, keep = A._c()
        self._chk(self._L.kl_lanczos(self._h, C.byref(o), nx, ny, steps, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def cheb_interval_from_ritz(self, theta_max: float, degree: int):
        """params for cheb(degree): (b, b/ratio(degree)) with b = 1.025*theta_max (kl_cheb_interval_from_ritz)."""
        out = (C.c_double * 2)()
        self._chk(self._L.kl_cheb_interval_from_ritz(theta_max, int(degree), out))
        return (out[0], out[1])

    def cheb_params_from_ritz(self, theta_min: float, theta_max: float):
        out = (C.c_double * 2)()
        self._L.kl_cheb_params_from_ritz(theta_min, theta_max, out)
        return (out[0], out[1])
