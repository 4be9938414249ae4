"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE -- not product code).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module.  Function names and argument order
follow the reference's Fortran module procedures (cited in krylov_oracle.c).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libkrylov_oracle.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
STENCIL_FN = C.CFUNCTYPE(None, _dp, _dp, C.c_int)
PRECOND_FN = C.CFUNCTYPE(None, STENCIL_FN, _dp, _dp, _dp, _dp, C.c_int, C.c_int64)


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("krylov_oracle.c", "krylov_extras.c", "Makefile")]
    if force or not os.path.exists(_SO) or any(
        os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs
    ):
        subprocess.check_call(["make", "-C", _HERE, "-B"], stdout=subprocess.DEVNULL)
    return _SO


_lib = None


_native_dir = None


def build_native() -> str:
    """A copy built with -march=native (the reference's own flag, CMakeLists.txt:5) on THIS machine, for timing
    the CPU baseline on the box it runs on.  The portable x86-64-v3 build stays the checker.  The copy goes to a
    temporary directory (removed at exit), so that the source tree may be read-only.  Returns the path (or the
    portable library's path if the compiler is missing)."""
    global _SO, _lib, _native_dir
    try:
        if _native_dir is None:
            _native_dir = tempfile.TemporaryDirectory(prefix="krylov_oracle_native_")
        so = os.path.join(_native_dir.name, "libkrylov_oracle.so")
        subprocess.check_call(
            ["gcc", "-O3", "-fopenmp", "-march=native", "-funroll-loops", "-ffp-contract=off", "-fPIC", "-std=gnu11",
             "-shared", "-o", so, os.path.join(_HERE, "krylov_oracle.c"), os.path.join(_HERE, "krylov_extras.c"), "-lm"],
            stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    except Exception:
        return build()
    _SO, _lib = so, None
    return so


def lib():
    global _lib
    if _lib is None:
        if _native_dir is None or not _SO.startswith(_native_dir.name):
            build()
        L = C.CDLL(_SO)
        for name in ("ko_get_stvec", "ko_get_stv_poisson", "ko_get_aniso"):
            getattr(L, name).restype = STENCIL_FN
        for name in ("ko_get_cbpr2", "ko_get_identity", "ko_get_cheb"):
            getattr(L, name).restype = PRECOND_FN
        L.ko_hh_orth_frobenius.restype = C.c_double
        L.ko_omp_max_threads.restype = C.c_int
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(_dp)


def set_threads(t: int):
    lib().ko_omp_set_threads(int(t))


def max_threads() -> int:
    return int(lib().ko_omp_max_threads())


# ---- operators / preconditioners (built-ins are C function pointers) ----
def stvec_fn():
    return lib().ko_get_stvec()


def stv_poisson_fn():
    return lib().ko_get_stv_poisson()


def aniso_fn(eps_x: float, eps_y: float):
    lib().ko_set_aniso(C.c_double(eps_x), C.c_double(eps_y))
    return lib().ko_get_aniso()


_aniso_var_keep = None


def aniso_var_fn(kx: np.ndarray, ky: np.ndarray):
    """variable-coefficient anisotropic diffusion (krylov_extras.c ko_aniso_var); kx, ky: cell coefficient grids"""
    global _aniso_var_keep
    kx = np.ascontiguousarray(kx, dtype=np.float64).reshape(-1)
    ky = np.ascontiguousarray(ky, dtype=np.float64).reshape(-1)
    _aniso_var_keep = (kx, ky)
    lib().ko_set_aniso_var(_p(kx), _p(ky))
    lib().ko_get_aniso_var.restype = STENCIL_FN
    return lib().ko_get_aniso_var()


def cbpr2_fn():
    return lib().ko_get_cbpr2()


def identity_fn():
    return lib().ko_get_identity()


def cheb_fn(degree: int):
    lib().ko_set_cheb_degree(int(degree))
    return lib().ko_get_cheb()


def apply(A, x: np.ndarray, nsize: int, parallel: bool = False) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    lib().ko_apply(A, _p(x), _p(y), int(nsize), int(parallel))
    return y


def apply_precond(M, A, r: np.ndarray, params, nsize: int, parallel: bool = False):
    r = np.ascontiguousarray(r, dtype=np.float64)
    z = np.zeros_like(r)
    aux = np.zeros_like(r)
    params = np.ascontiguousarray(params, dtype=np.float64)
    lib().ko_apply_precond(M, A, _p(r), _p(z), _p(aux), _p(params), int(nsize),
                           C.c_int64(r.size), int(parallel))
    return z


def manufactured_rhs(A, nsize: int) -> np.ndarray:
    b = np.zeros(nsize * nsize)
    lib().ko_manufactured_rhs(A, int(nsize), _p(b))
    return b


@dataclass
class GmresResult:
    x: np.ndarray
    final_err: np.ndarray
    v_err: np.ndarray
    n_out: int
    restart_out: int
    history: np.ndarray = field(default_factory=lambda: np.zeros(0))
    orth_frob: float = float("nan")

    @property
    def iterations(self) -> int:  # tests/test_poisson_mf.f90:78  (restart_out - 1) * m + n_out, m = size(final_err)
        return (self.restart_out - 1) * int(self.final_err.size) + self.n_out


@dataclass
class CgResult:
    x: np.ndarray
    iter: int
    res: float
    history: np.ndarray


def _hist(cap):
    h = np.zeros(max(cap, 1))
    hl = C.c_int(0)
    return h, hl


def gmres_mgsr_mf(Ax_vec, b, m, tol, M_inv, params, max_restarts=0, ortho=0, history_cap=200000):
    b = np.ascontiguousarray(b, dtype=np.float64)
    n = b.size
    x = np.zeros(n); fe = np.zeros(m); ve = np.zeros(m + 1)
    n_out = C.c_int(0); rs = C.c_int(0)
    params = np.ascontiguousarray(params, dtype=np.float64)
    h, hl = _hist(history_cap)
    rc = lib().ko_gmres_mgsr_mf(Ax_vec, _p(b), C.c_int64(n), _p(x), int(m), C.c_double(tol),
                                _p(fe), _p(ve), C.byref(n_out), C.byref(rs), M_inv, _p(params),
                                int(max_restarts), int(ortho), _p(h), int(history_cap), C.byref(hl))
    assert rc == 0
    return GmresResult(x, fe, ve, n_out.value, rs.value, h[: min(hl.value, history_cap)].copy())


def gmres_mgsr_omp(Ax_vec, b, m, tol, M_inv, params, max_restarts=0, ortho=0, skip_verr=False,
                   history_cap=200000):
    b = np.ascontiguousarray(b, dtype=np.float64)
    n = b.size
    x = np.zeros(n); fe = np.zeros(m); ve = np.zeros(m + 1)
    n_out = C.c_int(0); rs = C.c_int(0)
    params = np.ascontiguousarray(params, dtype=np.float64)
    h, hl = _hist(history_cap)
    rc = lib().ko_gmres_mgsr_omp(Ax_vec, _p(b), C.c_int64(n), _p(x), int(m), C.c_double(tol),
                                 _p(fe), _p(ve), C.byref(n_out), C.byref(rs), M_inv, _p(params),
                                 int(max_restarts), int(ortho), int(skip_verr), _p(h),
                                 int(history_cap), C.byref(hl))
    assert rc == 0
    return GmresResult(x, fe, ve, n_out.value, rs.value, h[: min(hl.value, history_cap)].copy())


def gmres_hh(Ax_vec, b, m, tol, M_inv=None, params=(0.0, 0.0), max_stages=0, skip_verr=False,
             want_orth=False, history_cap=200000):
    """M_inv None -> gmres_hh_omp (gmres_hh.f90:211); else gmres_hh_prec_omp (:388)."""
    b = np.ascontiguousarray(b, dtype=np.float64)
    n = b.size
    x = np.zeros(n); fe = np.zeros(m); ve = np.zeros(m + 1)
    n_out = C.c_int(0); st = C.c_int(0)
    params = np.ascontiguousarray(params, dtype=np.float64)
    h, hl = _hist(history_cap)
    orth = C.c_double(float("nan"))
    mi = M_inv if M_inv is not None else C.cast(None, PRECOND_FN)
    rc = lib().ko_gmres_hh(Ax_vec, _p(b), C.c_int64(n), _p(x), int(m), C.c_double(tol), _p(fe),
                           _p(ve), C.byref(n_out), C.byref(st), mi, _p(params), int(max_stages),
                           int(skip_verr), C.byref(orth) if want_orth else None, _p(h),
                           int(history_cap), C.byref(hl))
    assert rc == 0
    return GmresResult(x, fe, ve, n_out.value, st.value, h[: min(hl.value, history_cap)].copy(),
                       orth.value)


# ---- dense-operator variants (gmres_mgsr.f90:11, gmres_hh.f90:10, hilbert.f90:6) ----
_dense_keep = None


def dense_fn(A: np.ndarray):
    """A(n,n) as the Fortran array (column-major storage): pass a numpy array whose [i, j] is A(i,j)."""
    global _dense_keep
    Af = np.asfortranarray(A, dtype=np.float64)
    _dense_keep = Af
    lib().ko_set_dense(Af.ctypes.data_as(_dp), C.c_int64(Af.shape[0]))
    lib().ko_get_dense.restype = STENCIL_FN
    return lib().ko_get_dense()


def generate_matrix(n: int) -> np.ndarray:
    """hilbert::generate_matrix (single-precision reciprocals widened to double)."""
    H = np.zeros((n, n), order="F")
    lib().ko_generate_matrix(H.ctypes.data_as(_dp), int(n))
    return H


def dense_matvec(A: np.ndarray, x: np.ndarray) -> np.ndarray:
    f = dense_fn(A)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    f(_p(x), _p(y), 0)
    return y


def gmres_mgsr_dense(A, b, m, tol, max_restarts=0, history_cap=200000):
    """gmres_mgsr.f90:11-95 = the _mf algorithm on w = matmul(A, v) without preconditioner."""
    lib().ko_get_identity.restype = PRECOND_FN
    return gmres_mgsr_mf(dense_fn(A), b, m, tol, lib().ko_get_identity(), (0.0, 0.0), max_restarts, 0, history_cap)


def gmres_hh_dense(A, b, m, tol, max_stages=0, history_cap=200000):
    f = dense_fn(A)  # noqa: F841  (sets the global operator)
    b = np.ascontiguousarray(b, dtype=np.float64)
    n = b.size
    x = np.zeros(n); fe = np.zeros(m); ve = np.zeros(m + 1)
    n_out = C.c_int(0); st = C.c_int(0)
    h, hl = _hist(history_cap)
    rc = lib().ko_gmres_hh_dense(_p(b), C.c_int64(n), _p(x), int(m), C.c_double(tol), _p(fe), _p(ve),
                                 C.byref(n_out), C.byref(st), int(max_stages), _p(h), int(history_cap),
                                 C.byref(hl))
    assert rc == 0
    return GmresResult(x, fe, ve, n_out.value, st.value, h[: min(hl.value, history_cap)].copy())


def _cg_like(fn, A, b, tol, max_iter, M_inv, params, history_cap):
    b = np.ascontiguousarray(b, dtype=np.float64)
    n = b.size
    x = np.zeros(n)
    it = C.c_int(int(max_iter)); res = C.c_double(0.0)
    params = np.ascontiguousarray(params, dtype=np.float64)
    h, hl = _hist(history_cap)
    mi = M_inv if M_inv is not None else C.cast(None, PRECOND_FN)
    rc = fn(A, _p(b), C.c_int64(n), _p(x), C.c_double(tol), C.byref(it), C.byref(res), mi,
            _p(params), _p(h), int(history_cap), C.byref(hl))
    assert rc == 0
    return CgResult(x, it.value, res.value, h[: min(hl.value, history_cap)].copy())


def cg(A, b, tol, max_iter, history_cap=200000):
    return _cg_like(lib().ko_cg_serial, A, b, tol, max_iter, None, (0.0, 0.0), history_cap)


def pcg(A, b, tol, max_iter, M_inv, params, history_cap=200000):
    return _cg_like(lib().ko_cg_serial, A, b, tol, max_iter, M_inv, params, history_cap)


def cg_omp(A, b, tol, max_iter, history_cap=200000):
    return _cg_like(lib().ko_cg_omp, A, b, tol, max_iter, None, (0.0, 0.0), history_cap)


def pcg_omp(A, b, tol, max_iter, M_inv, params, history_cap=200000):
    return _cg_like(lib().ko_cg_omp, A, b, tol, max_iter, M_inv, params, history_cap)


def bicgstab(A, b, tol, max_iter, history_cap=200000):
    return _cg_like(lib().ko_bicgstab_serial, A, b, tol, max_iter, None, (0.0, 0.0), history_cap)


def pbicgstab(A, b, tol, max_iter, M_inv, params, history_cap=200000):
    return _cg_like(lib().ko_bicgstab_serial, A, b, tol, max_iter, M_inv, params, history_cap)


def pbicgstab_omp(A, b, tol, max_iter, M_inv, params, history_cap=200000):
    return _cg_like(lib().ko_pbicgstab_omp, A, b, tol, max_iter, M_inv, params, history_cap)


def lanczos_bounds(A, nsize: int, steps: int):
    """Extras (parity unpinned): k-step Lanczos on A from b = A*1 normalised."""
    out = np.zeros(2)
    alphas = np.zeros(steps); betas = np.zeros(steps)
    k = lib().ko_lanczos(A, int(nsize), int(steps), _p(out), _p(alphas), _p(betas))
    return float(out[0]), float(out[1]), alphas[:k].copy(), betas[:k].copy()
