"""ctypes loader of the CPU twin of KL_OP_STENCIL5 (tests/stencil5_twin.c; test infrastructure only).

The library is compiled on first use into a temporary directory (removed at exit), with the oracle's flags, so that
the source tree may be read-only.
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


def lib():
    global _lib, _dir
    if _lib is None:
        _dir = tempfile.TemporaryDirectory(prefix="stencil5_twin_")
        so = os.path.join(_dir.name, "libstencil5_twin.so")
        subprocess.check_call(["gcc", "-O3", "-fopenmp", "-march=x86-64-v3", "-funroll-loops", "-ffp-contract=off",
                               "-fPIC", "-std=gnu11", "-shared", "-o", so, os.path.join(_HERE, "stencil5_twin.c"),
                               "-lm"])
        _lib = C.CDLL(so)
        _lib.s5_set.argtypes = [C.c_double] * 5
    return _lib


def _p(a):
    return a.ctypes.data_as(_dp)


def set_weights(w):
    """w = (c, wl, wr, wd, wu)"""
    lib().s5_set(*[float(v) for v in w])


def apply_xy(w, x, nx, ny):
    """y = A(w) x on an nx x ny grid"""
    set_weights(w)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    lib().s5_apply_xy(_p(x), _p(y), int(nx), int(ny))
    return y


def stencil_fn(ko, w):
    """the twin as an operator of the oracle solvers and preconditioners (`ko` = oracle.oracle; square grids)"""
    set_weights(w)
    return ko.STENCIL_FN(C.cast(lib().s5_apply, C.c_void_p).value)


def dense(w, nx, ny):
    """the operator as a dense (nx*ny)^2 matrix, built from the weights (not from the twin)"""
    c, wl, wr, wd, wu = (float(v) for v in w)
    n = nx * ny
    A = np.zeros((n, n))
    for j in range(ny):
        for i in range(nx):
            k = i + j * nx
            A[k, k] = c
            if i > 0:
                A[k, k - 1] = -wl
            if i < nx - 1:
                A[k, k + 1] = -wr
            if j < ny - 1:
                A[k, k + nx] = -wd
            if j > 0:
                A[k, k - nx] = -wu
    return A
