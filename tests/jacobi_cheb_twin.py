"""ctypes loader of the CPU twin of KL_PC_JACOBI_CHEB (tests/jacobi_cheb_twin.c; test infrastructure only).

The library is compiled on first use into a temporary directory (removed at exit), with the oracle's flags, so that
the source tree may be read-only.  Coefficient fields are kept alive here while the twin holds pointers to them.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)
_lib = None
_dir = None
_keep = None


def lib():
    global _lib, _dir
    if _lib is None:
        _dir = tempfile.TemporaryDirectory(prefix="jacobi_cheb_twin_")
        so = os.path.join(_dir.name, "libjacobi_cheb_twin.so")
        subprocess.check_call(["gcc", "-O3", "-fopenmp", "-march=x86-64-v3", "-funroll-loops", "-ffp-contract=off",
                               "-fPIC", "-std=gnu11", "-shared", "-o", so, os.path.join(_HERE, "jacobi_cheb_twin.c"),
                               "-lm"])
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(_dp)


def set_fields(kx, ky):
    global _keep
    kx = np.ascontiguousarray(kx, dtype=np.float64).reshape(-1)
    ky = np.ascontiguousarray(ky, dtype=np.float64).reshape(-1)
    _keep = (kx, ky)
    lib().jc_set_fields(_p(kx), _p(ky))


def aniso_var_xy(kx, ky, x, nx, ny):
    """y = A(kx, ky) x on an nx x ny grid"""
    set_fields(kx, ky)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    lib().jc_aniso_var_xy(_p(x), _p(y), int(nx), int(ny))
    return y


def dinv(kx, ky, nx, ny):
    """1.0 / diag(A(kx, ky))"""
    set_fields(kx, ky)
    out = np.zeros(nx * ny)
    lib().jc_dinv_xy(_p(out), int(nx), int(ny))
    return out


def jacobi_cheb(kx, ky, r, degree, params, nx, ny):
    """z = M^-1 r of the given degree on an nx x ny grid"""
    set_fields(kx, ky)
    lib().jc_set_degree(int(degree))
    r = np.ascontiguousarray(r, dtype=np.float64)
    z = np.zeros_like(r)
    aux = np.zeros_like(r)
    prm = np.ascontiguousarray(params if len(params) else (0.0, 0.0), dtype=np.float64)
    lib().jc_jacobi_cheb_xy(_p(r), _p(z), _p(aux), _p(prm), int(nx), int(ny))
    return z


def precond_fn(ko, kx, ky, degree):
    """the twin as a preconditioner of the oracle solvers (`ko` = oracle.oracle; square grids)"""
    set_fields(kx, ky)
    lib().jc_set_degree(int(degree))
    return ko.PRECOND_FN(C.cast(lib().jc_precond, C.c_void_p).value)
